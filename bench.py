#!/usr/bin/env python
"""bench.py -- headline benchmark of the hot path (BASELINE.json): Mrays/s over all logical ray types and frame ms,
bun69k 4K (3840x2160) 16 spp, on N B200s, beside the CPU restatement of the reference on the host cores.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one full frame of the workload through the wavefront kernels.
  value    : whole-job throughput with the scene resident in HBM and the frame left on rank 0's device (NCCL chunk gather included for N>1)
  e2e      : same metric through the C ABI with HOST buffers: scene re-upload (H2D) on every rank + distributed render + frame read-back (D2H
             on rank 0) every step, wall clock between barriers, max over ranks -- the partitioned path, not N independent frames
  roofline : dominant kernel (k_trace): thread-instruction issue roofline.  achieved = closest-hit rays/s x I_ray, I_ray = I_fixed +
             node visits x I_node + triangle tests x I_prim with the per-ray counts MEASURED IN THIS RUN (counter build of the same kernels) and
             the instruction costs from profiles/sass/inst_model.json (tools/sass_model.py: SASS of the shipped build attributed to source
             regions by line info, dynamic counts from the committed ncu capture); peak = SMs x 4 schedulers x 32 lanes x SM clock of this run.
             Per rank at N>1.  compulsory_hbm and traffic (ncu DRAM bytes per launch) are printed beside it.
  cpu_baseline : the oracle ("port" of the reference; the Java reference cannot run here) on a bounded sample of the same workload
  --impl reference : the oracle on all host threads over a bounded WHOLE-FRAME sample (every 16th 8-row chunk); the GPU arm reports its rate
             on the same pixel set (`sample`), and checks that the pixels agree
N>1: one process per GPU (torchrun), frame split in interleaved 8-row chunks (strong scaling: the frame is fixed), chunks gathered to rank 0
by the library's own NCCL communicator (drt_comm_init / drt_render_distributed); torch.distributed only ships the communicator id and the timings.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # BASELINE.json configs[1] (the configuration the metric is quoted on): bun69k in the p3_t09 wrapper
    "bun69k": dict(scene="p3_t09.cli", cols=3840, rows=2160, spp=16, photons=-1, metric="Mrays/s (all ray types), bun69k 4K 16spp",
                   desc="configs[1]: bun69k in the p3_t09 wrapper; mesh = bun500 subdivided 3x, 61824 tris, stand-in for the missing bun69k.cli"),
    "t01": dict(scene="t01.cli", cols=3840, rows=2160, spp=16, photons=-1, metric="Mrays/s (all ray types), t01 4K 16spp", desc="configs[0]: two spheres, one point light"),
    "sierp": dict(scene="p3_t11_sierp.cli", cols=3840, rows=2160, spp=16, photons=-1, metric="Mrays/s (all ray types), p3_t11_sierp 4K 16spp",
                  desc="configs[2]: 21845 instances of the bun69k stand-in through the reference-topology instance BVH"),
    "planets": dict(scene="plnts3ColsBunnies.cli", cols=3840, rows=2160, spp=16, photons=-1, metric="Mrays/s (all ray types), plnts3ColsBunnies 4K 16spp",
                    desc="configs[3]: textured planets, bunny BVHs, reflection/refraction, spot + point lights"),
    "box_caustics": dict(scene="box_caustics.cli", cols=3840, rows=2160, spp=16, photons=4000000, metric="Mrays/s (all ray types incl. photon segments), box caustics 4K 16spp",
                         desc="configs[4]: Cornell wrapper around data/box.cli, caustic photon map k=80 r=0.05; photon pass inside every step"),
    "t11": dict(scene="t11.cli", cols=3840, rows=2160, spp=16, photons=1000000, metric="Mrays/s (all ray types incl. photon segments), t11 Cornell box 4K 16spp",
                desc="the reference scene behind its shipped box-caustics renders (t11c.png, boxCaustics*.png): Cornell box, mirror + glass spheres, point + disk light, diffuse photon map k=200 r=0.1"),
    "box_gi": dict(scene="box_gi.cli", cols=3840, rows=2160, spp=16, photons=1000000, metric="Mrays/s (all ray types incl. photon segments), box diffuse-GI 4K 16spp",
                   desc="configs[4] diffuse variant: diffuse photon map k=200 r=0.1; photon pass inside every step"),
}
WORKLOAD = dict(WORKLOADS["bun69k"])
METRIC = WORKLOAD["metric"]
CHUNK_ROWS = 8
SAMPLE_STRIDE = 16            # bounded CPU sample = every 16th 8-row chunk of the frame (the pixel set of rank 0 of 16)
ACCEL_NAMES = ["reference-topology literal", "reference-topology fast", "lbvh"]
DUMP_PIXELS = 1 << 21         # --dump-outputs: pixels kept of a larger frame (4 float32 channels + a float64 index: 48 MiB)


def make_config(w, world, accel, has_photons):
    """Identical in both arms (the driver compares them)."""
    return {"workload": "%s %dx%d %dspp%s (%s)" % (w["scene"], w["cols"], w["rows"], w["spp"], (", %d photons cast per light" % w["photons"]) if has_photons else "", w["desc"]),
            "accel": ACCEL_NAMES[accel], "l2": "flushed between timed iterations (256 MiB fill)",
            "partition": "interleaved %d-row chunks, NCCL send/recv gather to rank 0" % CHUNK_ROWS if world > 1 else "single GPU",
            "cpu_sample": "the CPU arms render every %dth %d-row chunk of the same frame (whole-frame sample); the GPU arm renders the whole frame and reports its rate on that pixel set as `sample`" % (SAMPLE_STRIDE, CHUNK_ROWS)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)), "measured"
    return {"hbm_gbs": 6650.0, "sm_max_mhz": 1965.0}, "fallback"


def source_hash():
    """Identity of the kernels' machine code (sha1 of the library's SASS, written by the build): the instruction model in profiles/sass/ is valid
    for the build it was derived from."""
    from distraytracer_old_b200 import build as B
    return B.kernel_hash()


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu, enabled=True):
        self.gpu, self.rows, self.stop, self.t, self.enabled = gpu, [], False, None, enabled

    def _run(self):
        while not self.stop:
            try:
                o = subprocess.run(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout.strip()
                if o:
                    self.rows.append([x.strip() for x in o.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def __enter__(self):
        if self.enabled:
            self.t = threading.Thread(target=self._run, daemon=True); self.t.start()
        return self

    def __exit__(self, *a):
        self.stop = True
        if self.t is not None:
            self.t.join(timeout=6)

    def summary(self):
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(self.rows)}


def dump_outputs(out_dir, frame_host, ray_types):
    """What the timed step hands its caller, as .npy files for comparing two builds output for output: the frame's A, R, G, B channels
    (float32; when the frame has more than DUMP_PIXELS pixels, the same seeded sample of them every run, their indices in frame_pixel_index)
    and the logical ray counts of the step (float64, in the order of ray_types_per_frame)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    n = frame_host.size
    idx = np.arange(n) if n <= DUMP_PIXELS else np.sort(np.random.default_rng(0).choice(n, DUMP_PIXELS, replace=False))
    px = frame_host.astype(np.uint32)[idx]
    np.save(os.path.join(out_dir, "frame_argb.npy"), np.stack([(px >> s) & 255 for s in (24, 16, 8, 0)], axis=1).astype(np.float32))
    np.save(os.path.join(out_dir, "frame_pixel_index.npy"), idx.astype(np.float64))
    np.save(os.path.join(out_dir, "ray_counts.npy"), np.array(list(ray_types.values()), dtype=np.float64))


def oracle_scene():
    from oracle import orc
    orc.build()
    w = WORKLOAD
    return orc.OracleScene(w["scene"], cols=w["cols"], rows=w["rows"], spp=w["spp"], photons=min(w["photons"], 200000) if w["photons"] >= 0 else -1)


def cpu_sample(o, threads, stride=SAMPLE_STRIDE, want_argb=False):
    r = o.render_chunks(CHUNK_ROWS, stride, 0, threads=threads, want_argb=want_argb)
    rays = sum(r["stats"][k] for k in ("primary", "shadow", "reflect", "refract"))
    return rays / r["seconds"] / 1e6, r["seconds"], rays, r["argb"]


def sample_text(threads, rays, stride=SAMPLE_STRIDE):
    w = WORKLOAD
    return "oracle (C++ restatement of the Java reference; no JDK on the box), %d thread%s, every %dth %d-row chunk of the %dx%d/%dspp frame = %d rays per step" % (
        threads, "" if threads == 1 else "s", stride, CHUNK_ROWS, w["cols"], w["rows"], w["spp"], rays)


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    o = oracle_scene()
    w = WORKLOAD
    secs, rays = [], 0
    for i in range(args.warmup + args.steps):
        v, s, rays, _ = cpu_sample(o, threads)
        if i >= args.warmup:
            secs.append(s)
    ms = 1e3 * sum(secs) / len(secs)
    value = rays / (ms / 1e3) / 1e6
    v1, s1, r1, _ = cpu_sample(o, 1, stride=SAMPLE_STRIDE * 8)            # the reference itself is single threaded (myScene.java:15 declares an unused executor)
    has_photons = w["photons"] >= 0
    print(json.dumps({"impl": "reference", "metric": METRIC, "value": round(value, 4), "unit": "Mrays/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                      "ms_per_step": round(ms, 3), "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                      "config": make_config(w, args.gpus, args.accel, has_photons),
                      "cpu_baseline": {"value": round(value, 4), "unit": "Mrays/s", "cores": threads, "kind": "port", "sample": sample_text(threads, rays),
                                       "single_thread": {"value": round(v1, 4), "unit": "Mrays/s", "cores": 1, "sample": sample_text(1, r1, SAMPLE_STRIDE * 8)}},
                      "e2e": {"value": round(value, 4), "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--accel", type=int, default=int(os.environ.get("DRT_ACCEL", "1")), help="0 reference-topology literal order, 1 reference-topology near-first (bit-identical results, default), 2 GPU LBVH")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg (profiling runs)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--workload", default="bun69k", choices=sorted(WORKLOADS) + ["synth"])
    ap.add_argument("--synth", default="soup:65536", help="with --workload synth: soup:N (N random triangles) or grid:K (K^3 bunny instances), see tools/make_synth.py")
    ap.add_argument("--photons", type=int, default=None, help="photons cast per light for the photon workloads (sweep 1M..64M)")
    ap.add_argument("--res", default=None, help="COLSxROWS override")
    ap.add_argument("--spp", type=int, default=None)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None, help="write the frame and ray counts of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    global METRIC
    if args.workload == "synth":
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        import make_synth
        kind, n = args.synth.split(":")
        path = getattr(make_synth, kind)(int(n)) if int(os.environ.get("RANK", "0")) == 0 or not os.path.exists(os.path.join(make_synth.GEN, "%s_%s.cli" % (kind, n))) else os.path.join(make_synth.GEN, "%s_%s.cli" % (kind, n))
        WORKLOADS["synth"] = dict(scene="gen/" + os.path.basename(path), cols=3840, rows=2160, spp=16, photons=-1, metric="Mrays/s (all ray types), synthetic %s 4K 16spp" % args.synth,
                                  desc="SURVEY 8(d) synthetic scaling scene %s under the config-2 camera and lights" % args.synth)
    WORKLOAD.clear(); WORKLOAD.update(WORKLOADS[args.workload]); METRIC = WORKLOAD["metric"]
    if args.photons is not None and WORKLOAD["photons"] >= 0:
        WORKLOAD["photons"] = args.photons
    if args.res:
        WORKLOAD["cols"], WORKLOAD["rows"] = (int(x) for x in args.res.lower().split("x"))
    if args.spp:
        WORKLOAD["spp"] = args.spp
    if args.impl == "reference":
        return reference_arm(args)
    args.warmup = max(args.warmup, 3)

    import numpy as np
    import torch
    import distraytracer_old_b200 as drt

    world = int(os.environ.get("WORLD_SIZE", "1")); rank = int(os.environ.get("RANK", "0")); local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dist = None
    w = WORKLOAD
    ctx = drt.Context(device=local, cols=w["cols"], rows=w["rows"])
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        # the library owns the data-path communicator; torch.distributed only ships its id (and, below, the timings)
        idt = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            idt.copy_(torch.frombuffer(bytearray(drt.Context.comm_unique_id()), dtype=torch.uint8))
        dist.broadcast(idt, 0)
        ctx.comm_init(bytes(idt.cpu().numpy().tobytes()), world, rank)
    scene = drt.Scene.from_cli(ctx, w["scene"], spp=w["spp"], photons=w["photons"], accel=args.accel)
    has_photons = scene.info()["photon_kind"] != 0
    npix = w["cols"] * w["rows"]
    n_chunks = (w["rows"] + CHUNK_ROWS - 1) // CHUNK_ROWS
    frame = torch.zeros(npix, dtype=torch.int32, device="cuda") if rank == 0 else None
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")      # > 126 MB L2
    torch.cuda.synchronize()                                               # the library works on its own stream: order it after torch's allocations / fills

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def step():
        # photon scenes: the reference emits the map inside draw() (myScene.initRender, :1096-1099), so the photon pass is part of every frame
        return scene.draw_distributed(dev_ptr=frame.data_ptr() if rank == 0 else None, chunk_rows=CHUNK_ROWS, reemit_photons=has_photons)

    for _ in range(args.warmup):
        flush.fill_(1); torch.cuda.synchronize(); step()
    barrier()
    gpu_ms, trace_ms, rays, launches = [], 0.0, 0, 0
    ray_types = None
    with ClockSampler(local, enabled=(rank == 0)) as cs:          # one sampler per job: concurrent nvidia-smi queries from every rank serialise on the driver
        for _ in range(args.steps):
            flush.fill_(1)                       # L2 flush between timed iterations
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            st = step()                          # returns after the library's stream has finished (rank 0: frame assembled)
            e1.record(); torch.cuda.synchronize()
            ms = e0.elapsed_time(e1)
            t = torch.tensor([ms, float(st.rays_total), float(st.kernel_launches), st.ms_trace, float(st.rays_primary), float(st.rays_shadow), float(st.rays_reflect),
                              float(st.rays_refract), float(st.rays_photon)], dtype=torch.float64, device="cuda")
            if dist is not None:
                mx = t.clone(); dist.all_reduce(mx, op=dist.ReduceOp.MAX); sm = t.clone(); dist.all_reduce(sm, op=dist.ReduceOp.SUM)
                ms, r, l, tr = mx[0].item(), sm[1].item(), sm[2].item(), mx[3].item()
                types = [sm[k].item() for k in range(4, 9)]          # every rank reports its own share (pixels of its chunks, photon indices of its range)
            else:
                r, l, tr = t[1].item(), t[2].item(), t[3].item(); types = [t[k].item() for k in range(4, 9)]
            gpu_ms.append(ms); rays = int(r); launches = int(l); trace_ms += tr
            ray_types = dict(zip(("primary", "shadow", "reflect", "refract", "photon_segments"), (int(x) for x in types)))
            stage = {"trace": st.ms_trace, "shade": st.ms_shade, "light": st.ms_light, "other": st.ms_other, "render_total": st.ms_total}
            rank_rays_closest = st.rays_primary + st.rays_reflect + st.rays_refract
    clocks = cs.summary()
    frame_crc = None
    if rank == 0:      # identical for every GPU count (sampler keyed by absolute pixel, canonical photon order)
        import zlib
        frame_host = frame.cpu().numpy()
        frame_crc = "%08x" % (zlib.crc32(frame_host.tobytes()) & 0xffffffff)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, frame_host, ray_types)
    ms_per_step = sum(gpu_ms) / len(gpu_ms)
    value = rays / (ms_per_step / 1e3) / 1e6

    # ---- e2e through the C ABI with host buffers: every rank re-uploads the scene (H2D), the partitioned frame is rendered and gathered, rank 0
    #      reads it back into pinned host memory (D2H).  Wall clock between barriers, max over ranks.
    e2e = None
    if not args.no_e2e:
        host = torch.empty(npix, dtype=torch.int32).pin_memory() if rank == 0 else None
        scene_bytes = scene.accel_info()["scene_bytes"]            # what drt_scene_reupload copies host -> device
        for _ in range(2):
            scene.reupload(); scene.draw_distributed(host_ptr=host.data_ptr() if rank == 0 else None, chunk_rows=CHUNK_ROWS, reemit_photons=has_photons)
        barrier(); t0 = time.perf_counter()
        for _ in range(args.steps):
            scene.reupload()                        # H2D of the flattened scene
            scene.draw_distributed(host_ptr=host.data_ptr() if rank == 0 else None, chunk_rows=CHUNK_ROWS, reemit_photons=has_photons)   # kernels + NCCL gather + D2H of the ARGB frame
        torch.cuda.synchronize(); dt = time.perf_counter() - t0
        if dist is not None:
            tt = torch.tensor([dt], dtype=torch.float64, device="cuda"); dist.all_reduce(tt, op=dist.ReduceOp.MAX); dt = tt.item()
        e2e = {"value": round(rays * args.steps / dt / 1e6, 3), "unit": "Mrays/s", "h2d_bytes_per_step": int(scene_bytes) * world, "d2h_bytes_per_step": npix * 4,
               "ms_per_step": round(1e3 * dt / args.steps, 3),
               "note": "every rank: drt_scene_reupload (H2D); drt_render_distributed: partitioned render + NCCL gather + D2H of the frame into pinned host memory on rank 0; wall clock, max over ranks"}
        if rank == 0:
            import zlib
            e2e["frame_crc32"] = "%08x" % (zlib.crc32(host.numpy().tobytes()) & 0xffffffff)

    # ---- the pixel set the CPU arms render (every 16th chunk), on this GPU: rate + pixel agreement
    sample = None; roof = None; cpu = None
    if rank == 0:
        sbuf = torch.zeros(npix, dtype=torch.int32, device="cuda"); torch.cuda.synchronize()
        for _ in range(2):
            sst = scene.draw_device_chunks(SAMPLE_STRIDE, 0, CHUNK_ROWS, sbuf.data_ptr())
        sample = {"value": round(sst.rays_total / (sst.ms_total / 1e3) / 1e6, 3), "unit": "Mrays/s", "rays": int(sst.rays_total), "ms": round(sst.ms_total, 3),
                  "pixels": "every %dth %d-row chunk (the reference arm's pixel set)" % (SAMPLE_STRIDE, CHUNK_ROWS)}

        # ---- roofline of the dominant kernel (k_trace): thread-instruction issue roofline, per rank
        peaks, which = measured_peaks()
        cctx = drt.Context(device=local, cols=max(16, w["cols"] // 8), rows=max(16, w["rows"] // 8), counters=True)          # same camera/scene at 1/8 linear size: per-ray averages
        cs2 = drt.Scene.from_cli(cctx, w["scene"], spp=w["spp"], photons=min(w["photons"], 100000) if w["photons"] >= 0 else -1, accel=args.accel)
        _, cst = cs2.draw()
        r_all = cst.rays_primary + cst.rays_reflect + cst.rays_refract          # rays traced by k_trace (closest hit)
        box_per_ray, prim_per_ray = cst.box_tests_closest / max(1, r_all), cst.prim_tests_closest / max(1, r_all)
        cctx.close()
        sm_mhz = clocks.get("sm_mhz") or peaks.get("sm_max_mhz", 1965.0)
        n_sm = torch.cuda.get_device_properties(local).multi_processor_count
        peak_inst = n_sm * 4 * 32 * sm_mhz * 1e6                                        # thread instructions / s
        ms_trace_step = trace_ms / len(gpu_ms)                                         # this rank's k_trace time per frame (max over ranks at N>1)
        model_path = os.path.join(ROOT, "profiles", "sass", "inst_model.json")
        model = json.load(open(model_path)) if os.path.exists(model_path) else None
        roof = {"bound": "issue", "kernel": "k_trace (lean variant + generic fix-up)", "unit": "Gthread-inst/s", "peak": round(peak_inst / 1e9, 1),
                "peak_source": "%d SMs x 4 schedulers x 32 lanes x %.0f MHz (SM clock sampled during the timed region)" % (n_sm, sm_mhz),
                "per_ray": {"box_tests": round(box_per_ray, 2), "node_visits": round(box_per_ray / 2, 2), "prim_tests": round(prim_per_ray, 2)},
                "ms_trace_per_step": round(ms_trace_step, 3), "rays_closest_per_step_this_rank": int(rank_rays_closest), "traffic": None}
        if model is not None:
            m = model["k_trace"]
            i_ray = m["I_fixed"] + (box_per_ray / 2) * m["I_node"] + prim_per_ray * m["I_prim"]
            achieved = rank_rays_closest * i_ray / (ms_trace_step / 1e3)
            roof.update({"achieved": round(achieved / 1e9, 1), "frac": round(achieved / peak_inst, 4),
                         "model": {"I_fixed": m["I_fixed"], "I_node": m["I_node"], "I_prim": m["I_prim"], "I_ray": round(i_ray, 1), "source": "profiles/sass/inst_model.json (tools/sass_model.py)",
                                   "derived_from_build": model.get("source_hash"), "this_build": source_hash(), "ncu_issue_slot_util_of_profiled_launch": m.get("ncu_issue_util"),
                                   "ncu_thread_inst_per_ray_of_profiled_launch": m.get("ncu_thread_inst_per_ray")}})
        else:
            roof.update({"achieved": None, "frac": None, "model": "profiles/sass/inst_model.json missing: run tools/sass_model.py on an ncu capture of this build"})
        # the same kernel against the bytes that MUST cross HBM (hit record out; primary rays are generated in the kernel, the scene is cache resident)
        compulsory = rank_rays_closest * 96.0 / (ms_trace_step / 1e3) / 1e9
        roof["compulsory_hbm"] = {"achieved": round(compulsory, 1), "unit": "GB/s", "peak": peaks["hbm_gbs"], "frac": round(compulsory / peaks["hbm_gbs"], 4), "bytes_per_ray": 96, "peak_source": which + " (burst copy)"}
        tr_path = os.path.join(ROOT, "profiles", "trace_traffic.json")
        if os.path.exists(tr_path):
            try:
                roof["traffic"] = json.load(open(tr_path)).get("dram_bytes_per_launch")
            except Exception:
                pass
        if world == 1 and not args.no_cpu:
            o = oracle_scene()
            threads = os.cpu_count() or 1
            v, secs, crays, cargb = cpu_sample(o, threads, want_argb=True)
            v1, s1, r1, _ = cpu_sample(o, 1, stride=SAMPLE_STRIDE * 8)
            # pixel agreement on the shared pixel set (photon workloads: the CPU leg casts fewer photons, so only non-photon workloads are compared)
            agree = None
            if not has_photons:
                g = sbuf.cpu().numpy().reshape(w["rows"], w["cols"])
                rows_idx = [c * CHUNK_ROWS + k for c in range(0, n_chunks, SAMPLE_STRIDE) for k in range(CHUNK_ROWS) if c * CHUNK_ROWS + k < w["rows"]]
                gs, cs_ = g[rows_idx], cargb[:len(rows_idx)]
                ch = lambda a, sh: ((a.astype(np.uint32) >> sh) & 255).astype(np.int32)
                d = np.maximum(np.maximum(np.abs(ch(gs, 16) - ch(cs_, 16)), np.abs(ch(gs, 8) - ch(cs_, 8))), np.abs(ch(gs, 0) - ch(cs_, 0)))
                agree = {"pixels": int(d.size), "frac_within_2_of_255": round(float((d <= 2).mean()), 6), "max_abs_diff": int(d.max())}
            cpu = {"value": round(v, 4), "unit": "Mrays/s", "cores": threads, "kind": "port", "sample": sample_text(threads, crays) + " in %.1f s" % secs,
                   "single_thread": {"value": round(v1, 4), "unit": "Mrays/s", "cores": 1, "sample": sample_text(1, r1, SAMPLE_STRIDE * 8) + " in %.1f s (the reference itself is single threaded)" % s1},
                   "gpu_pixels_agree": agree}

    if rank == 0:
        line = {"metric": METRIC, "value": round(value, 3), "unit": "Mrays/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms_per_step, 3),
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": make_config(w, world, args.accel, has_photons),
                "frame_ms": round(ms_per_step, 3), "frame_crc32": frame_crc, "rays_per_frame": rays, "ray_types_per_frame": ray_types, "accel_info": scene.accel_info(), "build_info": {k: (round(v, 2) if isinstance(v, float) else v) for k, v in scene.build_info().items()},
                "stages_ms_rank0_last_step": {k: round(v, 3) for k, v in stage.items()}, "gpu_launches": launches, "host_syncs_per_frame": int(st.host_syncs), "rays_deferred_to_generic_kernels": int(st.rays_deferred),
                "clocks": clocks, "e2e": e2e, "sample": sample, "roofline": roof, "cpu_baseline": cpu}
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier(); dist.destroy_process_group()
    ctx.close()


if __name__ == "__main__":
    main()
