#!/usr/bin/env python
"""Instruction model of the traversal kernels from SASS (SURVEY 8(d): I_ray = n_nodes * I_box + n_prims * I_prim + I_shade, "I_* counted from
SASS of the shipped kernels").

  python tools/sass_model.py --rep gpurun_out/prof.ncu-rep [--lib distraytracer_old_b200/libdrt.so] [--out profiles/sass]

What it does, for k_trace<false,0> and k_light<false,0> (the lean variants the benchmark scene runs) and for k_shade (one region: I_shade = I_fixed):
  1. extracts the sm_100a cubin of --lib and disassembles it with line info and inlining chains (nvdisasm -gi); the kernel's SASS is saved
     under --out for the record;
  2. attributes every SASS instruction to a source REGION: "node" = anything inlined from between the [sass:node-begin] / [sass:node-end]
     markers of csrc/dev_isect.cuh (one inner-node visit of the FP32 pre-test descent: 4 loads, 2 box tests, child selection, push / pop),
     "leaf" = between [sass:leaf-begin] / [sass:leaf-end] (the triangle loop of a leaf, FP64), "fixed" = everything else (ray generation or
     load, top-level loop, transforms, hit record) -- the STATIC counts;
  3. reads the per-instruction execution counts of the same kernel from the ncu report (--rep must have been captured from THIS build:
     the instruction sequences are matched one to one) and forms the DYNAMIC thread-level costs
        I_node  = thread instructions executed in "node" / thread-level node visits   (visits = executions of the node's first load)
        I_prim  = thread instructions executed in "leaf" / thread-level triangle tests (tests = executions of the triangle's first load)
        I_fixed = thread instructions executed in "fixed" / rays of the launch
     which is what bench.py multiplies with the per-ray node-visit and triangle-test counts it measures in its own run.
Writes <out>/inst_model.json (+ the source hash of the build, the launch's measured issue-slot utilisation and thread instructions per ray)."""
import argparse, csv, hashlib, io, json, os, re, subprocess, sys, tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
KERNELS = {"k_trace": r"_ZN3drt7k_traceILb0ELi0EEE", "k_light": r"_ZN3drt7k_lightILb0ELi0EEE", "k_shade": r"_ZN3drt7k_shadeILb1EEE"}   # k_shade<true>: level 0
VARIANT = {"k_trace": "<(bool)0, (int)0>", "k_light": "<(bool)0, (int)0>", "k_shade": "k_shade<(bool)1>"}      # launch name filter in the ncu report
RAWNAME = {"k_trace": "<0, 0>", "k_light": "<0, 0>", "k_shade": "k_shade<1>"}


def marker_ranges():
    src = open(os.path.join(ROOT, "distraytracer_old_b200", "csrc", "dev_isect.cuh")).read().splitlines()
    out = {"node": [], "leaf": []}
    open_ = {}
    for i, l in enumerate(src, 1):
        m = re.search(r"\[sass:(node|leaf)-(begin|end)\]", l)
        if m:
            if m.group(2) == "begin":
                open_[m.group(1)] = i
            else:
                out[m.group(1)].append((open_.pop(m.group(1)), i))
    return out


def disassemble(lib, mangled_prefix, workdir):
    subprocess.run(["cuobjdump", "-xelf", "all", os.path.abspath(lib)], cwd=workdir, check=True, capture_output=True)
    cubins = [f for f in os.listdir(workdir) if f.endswith(".cubin")]
    cubin = max(cubins, key=lambda f: os.path.getsize(os.path.join(workdir, f)))
    txt = subprocess.run(["nvdisasm", "-gi", "-c", os.path.join(workdir, cubin)], capture_output=True, text=True, check=True).stdout.splitlines()
    insts, on, chain = [], False, []
    pending = []
    for l in txt:
        if l.startswith("\t.section") or l.lstrip().startswith(".section"):
            on = (".text." + mangled_prefix) in l or re.search(r"\.text\." + mangled_prefix, l) is not None
            continue
        if not on:
            continue
        m = re.search(r'//## File "([^"]+)", line (\d+)', l)
        if m:
            pending.append((os.path.basename(m.group(1)), int(m.group(2))))
            continue
        m = re.match(r"\s+/\*([0-9a-f]+)\*/\s+(.*?);", l)
        if m:
            if pending:
                chain = pending
                pending = []
            insts.append({"off": int(m.group(1), 16), "text": m.group(2).strip(), "chain": list(chain)})
    return insts


def region_of(inst, ranges):
    for kind in ("leaf", "node"):
        for f, line in inst["chain"]:
            if f == "dev_isect.cuh" and any(a <= line <= b for a, b in ranges[kind]):
                return kind
    return "fixed"


def ncu_rows(rep, name_regex, page, extra=()):
    r = subprocess.run(["ncu", "-i", rep, "--page", page, "--csv", "--kernel-name", "regex:" + name_regex, "--launch-count", "1"] + list(extra), capture_output=True, text=True)
    return list(csv.reader(io.StringIO(r.stdout)))


def source_hash():
    """sha1 of the library's SASS (distraytracer_old_b200/build.py: kernel_hash): host-side edits do not change it, any kernel change does"""
    from distraytracer_old_b200 import build as B
    return B.kernel_hash()


def opcode(text):
    t = text.split()
    if t and t[0].startswith("@"):
        t = t[1:]
    return t[0] if t else ""


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rep", required=True)
    ap.add_argument("--lib", default=os.path.join(ROOT, "distraytracer_old_b200", "libdrt.so"))
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "sass"))
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    ranges = marker_ranges()
    model = {"source_hash": source_hash(), "marker_lines": ranges, "ncu_report": os.path.basename(a.rep)}
    for kname, mangled in KERNELS.items():
        with tempfile.TemporaryDirectory() as wd:
            insts = disassemble(a.lib, mangled, wd)
        with open(os.path.join(a.out, kname + ("_lean.sass" if kname != "k_shade" else ".sass")), "w") as f:
            for i in insts:
                f.write("/*%04x*/ %-70s // %s %s\n" % (i["off"], i["text"][:70], region_of(i, ranges), " <- ".join("%s:%d" % c for c in i["chain"][:2])))
        static = {"node": 0, "leaf": 0, "fixed": 0}
        for i in insts:
            static[region_of(i, ranges)] += 1
        entry = {"static_instructions": static, "sass_file": kname + ("_lean.sass" if kname != "k_shade" else ".sass")}
        rows = ncu_rows(a.rep, kname + "<.*0, .*0>" if False else kname, "source")
        # first kernel block whose name holds the lean variant
        hdr, data, take = None, [], False
        for r in rows:
            if r and r[0] == "Kernel Name":
                take = (VARIANT[kname] in r[1]) and not data
                continue
            if r and r[0] == "Address":
                hdr = r
                continue
            if take and hdr and len(r) == len(hdr):
                data.append(r)
        if data and len(data) == len(insts) and all(opcode(d[1]) == opcode(i["text"]) for d, i in zip(data, insts)):
            ci = {h: k for k, h in enumerate(hdr)}
            dyn = {"node": 0, "leaf": 0, "fixed": 0}
            first_load = {"node": 0, "leaf": 0}
            for d, i in zip(data, insts):
                reg = region_of(i, ranges)
                t = int(d[ci["Thread Instructions Executed"]])
                dyn[reg] += t
                if reg in first_load and opcode(i["text"]).startswith("LDG"):
                    first_load[reg] = max(first_load[reg], t)
            rays = max(int(d[ci["Thread Instructions Executed"]]) for d in data[:8])       # every thread of the launch executes the prologue
            raw = ncu_rows(a.rep, kname, "raw")
            rh = raw[0]
            rr = [r for r in raw[2:] if RAWNAME[kname] in r[rh.index("Kernel Name")]][0]
            # warp-level instructions x average active lanes (the full set does not carry the thread-level sum itself)
            total_thread = float(rr[rh.index("smsp__inst_executed.sum")]) * float(rr[rh.index("smsp__thread_inst_executed_per_inst_executed.ratio")])
            entry.update({"dynamic_thread_instructions": dyn, "thread_node_visits": first_load["node"], "thread_prim_tests": first_load["leaf"], "rays_of_profiled_launch": rays,
                          "I_node": round(dyn["node"] / max(1, first_load["node"]), 2), "I_prim": round(dyn["leaf"] / max(1, first_load["leaf"]), 2), "I_fixed": round(dyn["fixed"] / max(1, rays), 1),
                          "ncu_thread_inst_per_ray": round(total_thread / max(1, rays), 1), "ncu_issue_util": round(float(rr[rh.index("sm__inst_issued.avg.pct_of_peak_sustained_active")]) / 100, 4),
                          "ncu_time_ms": float(rr[rh.index("gpu__time_duration.sum")]), "node_visits_per_ray_profiled": round(first_load["node"] / max(1, rays), 3),
                          "prim_tests_per_ray_profiled": round(first_load["leaf"] / max(1, rays), 3)})
        else:
            entry["error"] = "ncu report does not match this build's SASS (%d profiled vs %d disassembled instructions): capture it again from this build" % (len(data), len(insts))
        model[kname] = entry
    json.dump(model, open(os.path.join(a.out, "inst_model.json"), "w"), indent=1)
    print(json.dumps({k: {x: v.get(x) for x in ("static_instructions", "I_node", "I_prim", "I_fixed", "ncu_thread_inst_per_ray", "ncu_issue_util", "error")} for k, v in model.items() if isinstance(v, dict) and "static_instructions" in v}, indent=1))


if __name__ == "__main__":
    main()
