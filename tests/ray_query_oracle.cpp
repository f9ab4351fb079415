// Test infrastructure for tests/test_gpu_ray_query.py: the CPU oracle's answers to explicit-ray queries.  Compiled by that test into a
// temporary directory against the oracle's headers (oracle/orc_scene.hpp), with the flags of oracle/Makefile; never part of the product.
//   rq_query_rays   Scene::findClosestRayHit per ray (as orc_trace_rays), plus the values the oracle shades a hit with: the world hit
//                   point RayHit::fwdTransHitLoc and the unit normal RayHit::objNorm (set by Geom::objHit / RayHit::reCalcCTMHitNorm)
//   rq_shadow_rays  Scene::calcShadow (myScene.java:879-885) per ray
// Rays are built as orc_trace_rays builds them (Ray(scene, org, dir, gen 0, default key)): their time comes from the sampler, so scenes with
// moving spheres are not compared.
#include "orc_scene.hpp"

using namespace orc;

extern "C" {

void* rq_load(const char* scene_file, const char* data_dir, const char* tex_dir, char* err, int errlen) {
  try {
    Options opt; opt.dataDir = data_dir; opt.texDir = tex_dir;
    Scene* s = new Scene(opt); s->readRTFile(scene_file, true);
    return s;
  } catch (std::exception& e) { if (err && errlen > 0) { strncpy(err, e.what(), errlen - 1); err[errlen - 1] = 0; } return nullptr; }
}
// ids2 = {primSerial, instSerial}, t, pos3, nrm3 (-1 / 0 on a miss).  Returns -1 if a winning hit does not carry its CTM and object.
int rq_query_rays(void* sv, long long n, const double* org, const double* dir, int32_t* ids, double* tOut, double* pos, double* nrm) {
  Scene* s = (Scene*)sv;
  for (long long i = 0; i < n; ++i) {
    SKey k; Ray r(s, Vec3(org[3 * i], org[3 * i + 1], org[3 * i + 2]), Vec3(dir[3 * i], dir[3 * i + 1], dir[3 * i + 2]), 0, k);
    RayHit h = s->findClosestRayHit(r);
    if (h.isHit && (!h.ctm || !h.obj)) return -1;
    ids[2 * i] = h.isHit ? h.obj->primSerial : -1; ids[2 * i + 1] = h.isHit ? h.instSerial : -1; tOut[i] = h.isHit ? h.t : 0;
    const Vec3 z(0, 0, 0), p = h.isHit ? h.fwdTransHitLoc : z, q = h.isHit ? h.objNorm : z;
    pos[3 * i] = p.x; pos[3 * i + 1] = p.y; pos[3 * i + 2] = p.z; nrm[3 * i] = q.x; nrm[3 * i + 1] = q.y; nrm[3 * i + 2] = q.z;
  }
  return 0;
}
// occluded[i] = 1 when something is hit with (dist - t) > EPS
int rq_shadow_rays(void* sv, long long n, const double* org, const double* dir, const double* dist, uint8_t* occluded) {
  Scene* s = (Scene*)sv;
  for (long long i = 0; i < n; ++i) {
    SKey k; Ray r(s, Vec3(org[3 * i], org[3 * i + 1], org[3 * i + 2]), Vec3(dir[3 * i], dir[3 * i + 1], dir[3 * i + 2]), 0, k);
    occluded[i] = s->calcShadow(r, dist[i]) == 1 ? 1 : 0;
  }
  return 0;
}

}  // extern "C"
