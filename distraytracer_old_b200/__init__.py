"""distraytracer_old_b200 -- B200-native wavefront renderer behind the render path of
jturner65/distRayTracer_old (package rayTracerDistAccelShdPhtnMap).

The product is `libdrt.so` (hand-written sm_100a CUDA kernels + C++ host interpreter + C ABI, see
include/drt.h).  This package is the thin Python host over that C ABI, mirroring the reference's own
interface for the path:

    reference                                       here
    ---------------------------------------------   -----------------------------------------
    myRTFileReader.readRTFile(file, null)           RTFileReader(ctx).readRTFile(file)  / Scene.from_cli
    one `switch` per .cli line (java :47-346)       Scene.command(line)
    `write` -> myScene.draw()  (java :86-93)        Scene.draw()  -> ARGB ints == PImage.pixels
    PImage.save                                     Scene.save(path)

Scene.intersect / Scene.occluded answer closest-hit and occlusion queries for the caller's own rays on CUDA tensors.

There is no CPU fallback: without the built library or without a CUDA device every render call raises.
"""
from .host import Context, Scene, Stats, RTFileReader, DrtError, lib_path, load_library, refine_steps, refine_pass, SCENES_DIR, ACCEL_REFERENCE, ACCEL_REFERENCE_FAST, ACCEL_LBVH  # noqa: F401
