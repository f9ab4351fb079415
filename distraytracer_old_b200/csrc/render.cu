// Wavefront renderer for sm_100a: ray generation, closest-hit trace, surface shading with secondary-ray enqueue
// (warp-aggregated atomic compaction), light/shadow pass, bottom-up bounce resolve, pixel resolve.
//
// Replaces the reference's recursive per-pixel loop (reference file:line, /root/reference/src/rayTracerDistAccelShdPhtnMap/):
//   k_raygen   myScene.java:1447-1462 (jittered AA), :1386-1406 + :868-875 (depth of field), :1563-1585 (fisheye), :1687-1701 (ortho),
//              single-sample loops :1498-1508, :1606-1625, :1723-1733
//   k_trace    myScene.java:888-903 findClosestRayHit (+ everything under it, see dev_isect.cuh)
//   k_shade    myScene.java:907-914 reflectRay, :1104-1149 skydome ; myObjShader.java:409-438 / :635-651 getColorAtPos (ambient, texture,
//              photon term, secondary rays :157-294, :503-631)
//   k_light    myObjShader.java:98-153 calcShadowColor ; myLight.java:33-41,77-82,159-163,251-266 ; myScene.java:879-885 calcShadow
//   k_resolve  the return path of the recursion: per-bounce clamp (myObjShader.java:661) then weighting (SURVEY Q14)
//   k_finish   mean of clamped samples, clamp, (int)(c*255) pack (myScene.java:1460, myObjShader.java:671)
#include "renderer.h"
#include "dbuf.h"
#include "dev_shade.cuh"
#include <cstdio>
#include <initializer_list>
#include <stdexcept>
#include <vector>

namespace drt {

// the device error word (dev_isect.cuh): devErrorFetch queues its copy to *e, which holds it after the next sync of `st`
static void devErrorReset(cudaStream_t st) { const unsigned int z = 0; CK(cudaMemcpyToSymbolAsync(g_devError, &z, sizeof(z), 0, cudaMemcpyHostToDevice, st)); }
static void devErrorFetch(unsigned int* e, cudaStream_t st) { CK(cudaMemcpyFromSymbolAsync(e, g_devError, sizeof(*e), 0, cudaMemcpyDeviceToHost, st)); }
static void throwIfIncomplete(unsigned int e) {
  if (e & DEV_ERR_INCOMPLETE) throw std::runtime_error("device search beyond its capacity (traversal stack overflow, or a photon query with more candidate ranges than the gather holds): the result would be incomplete");
}
static void devErrorCheck(cudaStream_t st) { unsigned int e = 0; devErrorFetch(&e, st); CK(cudaStreamSynchronize(st)); throwIfIncomplete(e); }

struct alignas(16) RayRec { double o[3], d[3]; double kt0, kt1; uint32_t ka, kb, kc, stream; int32_t gen, valid; int32_t pad[2]; };
struct alignas(16) SurfRec { double loc[3], n[3], rawDir[3], tex[3]; int32_t shader, valid; uint32_t ka, kb, kc, stream; int32_t gen, pad; };
struct alignas(16) NodeRec { double local[3], cA[3], cB[3], w[3]; int32_t parent, slot; int32_t pad[2]; };

// compact pixel index -> absolute pixel (row-major). Identity for single-GPU; interleaved row chunks for multi-GPU tiles.
// narrow != 0: the host checked that every ray index, pixel index and absolute pixel of the launch is below 2^31 (see renderChunks)
struct PixMap { long long chunkPix, totalPix; int world, rank, narrow; };
__host__ __device__ __forceinline__ long long absPixel(const PixMap& m, long long p) { return ((p / m.chunkPix) * m.world + m.rank) * m.chunkPix + (p % m.chunkPix); }

// primaryS / shadowS: the two counters every warp bumps are spread over 64 slots (block index & 63) and summed on the host -- one address for
// four million warps per frame showed up as 13 % of k_shade's stall samples.
// The first block accumulates over a whole render call; everything from `levelCount` on is the per-batch wavefront state (zeroed per batch):
// the number of rays of every bounce level and the lengths of the deferral lists live on the DEVICE, so the host never waits for a level.
#define DRT_MAX_LEVELS 16
struct Counters {
  unsigned long long primary, shadow, reflect, refract, box, prim, nextCount, boxC, primC, pad; unsigned long long primaryS[64], shadowS[64];
  unsigned long long deferredTotal, maxLevel;
  unsigned long long levelCount[DRT_MAX_LEVELS + 1], deferTrace[DRT_MAX_LEVELS + 1], deferLight[DRT_MAX_LEVELS + 1];
};
// wavefront geometry of one launch: level 0 holds n0 primary rays generated on the fly (no ray records), level L >= 1 holds levelCount[L]
// rays that level L-1's surface pass enqueued.  Node records of all levels of a batch are contiguous: level L starts at sum(levelCount[0..L-1]).
struct Wave { long long n0, rayCap, nodeCap; int level, launchedLevels; };
// (an overflowing level -- flagged, the frame is rendered again -- still has its counter bumped by every warp: clamp what is processed to what
// was actually stored, min(queue capacity, rest of the node pool), cumulatively over the levels below)
__device__ __forceinline__ long long waveNodeOffset(const Wave& w, const Counters* ctr, int level) {
  long long off = 0;
  for (int l = 0; l < level; ++l) { long long c = (long long)ctr->levelCount[l]; if (l > 0) { if (c > w.rayCap) c = w.rayCap; if (c > w.nodeCap - off) c = w.nodeCap - off; } off += c; }
  return off;
}
__device__ __forceinline__ long long waveCount(const Wave& w, const Counters* ctr) {
  if (w.level == 0) return w.n0;
  long long c = (long long)ctr->levelCount[w.level]; const long long room = w.nodeCap - waveNodeOffset(w, ctr, w.level);
  if (c > w.rayCap) c = w.rayCap; if (c > room) c = room; return c;
}

// Streaming (evict-first) access to the 16-byte-aligned wavefront records, field by field through registers: taking the address of a record
// variable (a generic memcpy) would pin the whole record in local memory for the lifetime of the kernel.
__device__ __forceinline__ int4 packDD(double a, double b) { return make_int4(__double2loint(a), __double2hiint(a), __double2loint(b), __double2hiint(b)); }
__device__ __forceinline__ double lo64(const int4& v) { return __hiloint2double(v.y, v.x); }
__device__ __forceinline__ double hi64(const int4& v) { return __hiloint2double(v.w, v.z); }
__device__ __forceinline__ void loadRayRec(RayRec& r, const RayRec* __restrict__ src) {
  const int4* q = reinterpret_cast<const int4*>(src);
  const int4 a = __ldcs(q), b = __ldcs(q + 1), c = __ldcs(q + 2), d = __ldcs(q + 3), e = __ldcs(q + 4), f = __ldcs(q + 5);
  r.o[0] = lo64(a); r.o[1] = hi64(a); r.o[2] = lo64(b); r.d[0] = hi64(b); r.d[1] = lo64(c); r.d[2] = hi64(c); r.kt0 = lo64(d); r.kt1 = hi64(d);
  r.ka = (uint32_t)e.x; r.kb = (uint32_t)e.y; r.kc = (uint32_t)e.z; r.stream = (uint32_t)e.w; r.gen = f.x; r.valid = f.y; r.pad[0] = f.z; r.pad[1] = f.w;
}
__device__ __forceinline__ void storeHit(Hit* __restrict__ dst, const Hit& h) {
  int4* d = reinterpret_cast<int4*>(dst);
  __stcs(d, make_int4(__double2loint(h.t), __double2hiint(h.t), h.prim, h.arg0));
  __stcs(d + 1, make_int4(h.arg1, h.state, h.hitXform, h.shaderOverride));
  __stcs(d + 2, make_int4(h.inst, h.pad0, __double2loint(h.loc.x), __double2hiint(h.loc.x)));
  __stcs(d + 3, packDD(h.loc.y, h.loc.z)); __stcs(d + 4, packDD(h.rawDir.x, h.rawDir.y)); __stcs(d + 5, packDD(h.rawDir.z, h.pad1));
}
static_assert(sizeof(RayRec) == 96 && sizeof(Hit) == 96, "record layout");
__device__ __forceinline__ void warpAdd(unsigned long long* dst, unsigned long long v) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  if ((threadIdx.x & 31) == 0 && v) atomicAdd(dst, v);
}
// warp-aggregated append of the calling lanes' indices to a deferral list
__device__ __forceinline__ void deferAppend(bool doIt, uint32_t idx, unsigned long long* counter, uint32_t* __restrict__ list) {
  const unsigned m = __ballot_sync(0xffffffffu, doIt); if (!m) return;
  const unsigned lane = threadIdx.x & 31; const int leader = __ffs(m) - 1;
  unsigned long long base = 0; if ((int)lane == leader) base = atomicAdd(counter, (unsigned long long)__popc(m));
  base = __shfl_sync(0xffffffffu, base, leader);
  if (doIt) list[base + __popc(m & ((1u << lane) - 1u))] = idx;
}

// ---------------------------------------------------------------------------------------------------------------
// absolute pixel and sample of primary-ray index i of the batch.  With pm.narrow the divisions run on 32-bit integers (a 64-bit division is a
// long subroutine, and there are up to four per ray): the same quotients, since every operand fits
struct PixKey { long long pix; uint32_t smp; };
__device__ __forceinline__ PixKey pixelOf(const FGlobals& g, const PixMap& pm, long long pix0, long long i) {
  const int spp = g.spp < 1 ? 1 : g.spp; PixKey k;
  if (pm.narrow) {
    const uint32_t ii = (uint32_t)i, p = (uint32_t)pix0 + ii / (uint32_t)spp, c = (uint32_t)pm.chunkPix;
    k.pix = (pm.world == 1) ? p : ((p / c) * (uint32_t)pm.world + (uint32_t)pm.rank) * c + p % c; k.smp = ii % (uint32_t)spp;
  } else { k.pix = absPixel(pm, pix0 + i / spp); k.smp = (uint32_t)(i % spp); }
  return k;
}
// primary ray of (pixel, sample) index i of the batch -- generated where it is needed (k_trace; k_shade only for a skydome miss) instead of
// being written to and re-read from HBM
__device__ __forceinline__ void primaryRay(const DScene& S, const PixMap& pm, long long pix0, long long i, RayRec& r) {
  const FGlobals& g = S.g; int spp = g.spp < 1 ? 1 : g.spp;
  const PixKey k = pixelOf(g, pm, pix0, i); const long long pix = k.pix; const uint32_t smp = k.smp;
  int row, col;
  if (pm.narrow) { row = (int)((uint32_t)pix / (uint32_t)g.cols); col = (int)((uint32_t)pix % (uint32_t)g.cols); }
  else { row = (int)(pix / g.cols); col = (int)(pix % g.cols); }
  r.kt0 = 1; r.kt1 = 1; r.ka = (uint32_t)pix; r.kb = smp; r.kc = 1; r.stream = STREAM_PIXEL; r.gen = 0; r.valid = 1; r.pad[0] = r.pad[1] = 0;
  D3 o = d3(g.eye[0], g.eye[1], g.eye[2]), d = d3(0, 0, -1);
  auto U = [&](uint32_t dim) { return philoxU01(g.seed, STREAM_PIXEL, (uint32_t)pix, smp, 1, dim); };
  if (g.spp < 1 || pix >= pm.totalPix) r.valid = 0;     // rays_per_pixel 0: the reference averages nothing (0/0 -> NaN -> 0); ragged last chunk
  if (g.camKind == CAM_FOV) {
    double rayY = (-1 * (row - g.rayYOffset)), rayX = col - g.rayXOffset;
    if (g.hasDof) {
      D3 lensCtr = norm3(d3(rayX, rayY, g.viewZ));
      // focal point: un-jittered pixel ray against plane z = -focalD  (N = (0,0,1), D = focalD)
      double planeRes = lensCtr.z, tf = -(((0 * o.x) + (0 * o.y)) + (1 * o.z) + g.focalD) / planeRes;
      D3 focal = d3((lensCtr.x * tf) + o.x, (lensCtr.y * tf) + o.y, (lensCtr.z * tf) + o.z);
      D3 tmp = norm3(rotAboutAxis(d3(0, 1, 0), d3(0, 0, -1), urange(U(DIM_LENS_ANGLE), 0, DRT_TWO_PI_F)));
      tmp = scale3(tmp, urange(U(DIM_LENS_RADIUS), 0, g.lensRadius)); o = add3(tmp, lensCtr);
      d = d3(focal.x - o.x, focal.y - o.y, focal.z - o.z);
    } else if (spp == 1) d = d3(rayX, rayY, g.viewZ);
    else { double ry = rayY + urange(U(DIM_AA_Y), -.5, .5), rx = rayX + urange(U(DIM_AA_X), -.5, .5); d = d3(rx, ry, g.viewZ); }
  } else if (g.camKind == CAM_FISHEYE) {
    double yVal, xVal;
    if (spp == 1) { yVal = (row + g.yStart) * g.fishMult; xVal = (col + g.xStart) * g.fishMult; }
    else { yVal = ((row + g.yStart) + urange(U(DIM_AA_Y), -.5, .5)) * g.fishMult; xVal = ((col + g.xStart) + urange(U(DIM_AA_X), -.5, .5)) * g.fishMult; }
    double rSq = (spp == 1) ? (xVal * xVal + yVal * yVal) : (yVal * yVal + xVal * xVal);
    if (rSq > 1) r.valid = 0;
    else { double rr = sqrt(rSq), theta = rr * g.aperatureHlf, phi = atan2(-yVal, xVal), sTh = sin(theta); d = d3(sTh * cos(phi), sTh * sin(phi), -cos(theta)); }
  } else {
    double ryo = g.rows / 2.0, rxo = g.cols / 2.0;
    if (spp == 1) o = d3(g.orthPerCol * (col - rxo), g.orthPerRow * (-1 * (row - ryo)), 0);
    else { double yB = g.orthPerRow * ((-1 * (row - ryo)) - .5), xB = g.orthPerCol * (col - rxo - .5);
      double ry = yB + (g.orthPerRow * urange(U(DIM_AA_Y), -.5, .5)), rx = xB + (g.orthPerCol * urange(U(DIM_AA_X), -.5, .5)); o = d3(rx, ry, 0); }
    d = d3(0, 0, -1);
  }
  d = norm3(d);
  r.o[0] = o.x; r.o[1] = o.y; r.o[2] = o.z; r.d[0] = d.x; r.d[1] = d.y; r.d[2] = d.z;
}

__device__ __forceinline__ double rayTime(const DScene& S, uint32_t stream, uint32_t a, uint32_t b, uint32_t c, uint32_t dim) {
  return S.g.pad0 ? philoxU01(S.g.seed, stream, a, b, c, dim) : 0.0;      // pad0 = scene has moving spheres
}

#ifndef DRT_TRACE_MINBLOCKS
#define DRT_TRACE_MINBLOCKS 5
#endif
#ifndef DRT_LIGHT_MINBLOCKS
#define DRT_LIGHT_MINBLOCKS 6
#endif
#ifndef DRT_LTRACE_MINBLOCKS
#define DRT_LTRACE_MINBLOCKS 6       // lean variants (F != TF_ALL)
#endif
#ifndef DRT_LLIGHT_MINBLOCKS
#define DRT_LLIGHT_MINBLOCKS 6
#endif
#ifndef DRT_L1_MINBLOCKS
#define DRT_L1_MINBLOCKS 6           // lean variants for scenes with instanced meshes (F == TF_LITERAL1)
#endif
// __launch_bounds__ min-blocks of the closest-hit kernels (k_trace, k_query_closest) and the shadow-ray kernels (k_light, k_query_any)
constexpr int traceMinBlocks(int F) { return (F == TF_ALL) ? DRT_TRACE_MINBLOCKS : (F == TF_LITERAL1) ? DRT_L1_MINBLOCKS : DRT_LTRACE_MINBLOCKS; }
constexpr int lightMinBlocks(int F) { return (F == TF_ALL) ? DRT_LIGHT_MINBLOCKS : (F == TF_LITERAL1) ? DRT_L1_MINBLOCKS : DRT_LLIGHT_MINBLOCKS; }

// The query kernels' loop over the rays of a launch (F: dev_isect.cuh).  Direct launch (work == null): rays [0, n).  Fix-up launch (the
// generic kernel, work != null): the *deferCount rays listed in `work`, counted once into Counters::deferredTotal.  body(i) returns whether
// ray i is deferred; a lean variant appends those, warp-collectively, to deferOut / *deferCount, which its fix-up launch reads.  The bodies
// are always_inline lambdas (optimised on their own first, they spill more).  k_trace / k_light write this loop out: through it they ran slower.
template <int F, class Body>
__device__ __forceinline__ void rayLoop(long long n, const uint32_t* work, unsigned long long* deferCount, uint32_t* deferOut, Counters* ctr, Body body) {
  if (work) n = (long long)*deferCount;
  if (work && n > 0 && blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(&ctr->deferredTotal, (unsigned long long)n);
  for (long long base = (long long)blockIdx.x * blockDim.x; base < n; base += (long long)gridDim.x * blockDim.x) {
    long long i = base + threadIdx.x; bool defer = false;
    if (i < n) {
      if (work) i = work[i];
      defer = body(i);
    }
    if (F != TF_ALL) deferAppend(defer, (uint32_t)i, deferCount, deferOut);
  }
}

// Closest-hit pass of one level.  F = compile-time feature set (dev_isect.cuh): the lean variants defer what they cannot serve to `deferOut`;
// the generic variant (TF_ALL) serves everything and is also the fix-up pass over such a list (`work` != null: ray indices to trace).
// rays == null: level 0, the primary ray is generated from the index.
template <bool COUNT, int F>
__global__ void __launch_bounds__(128, traceMinBlocks(F))
k_trace(const __grid_constant__ DScene S, Wave w, PixMap pm, long long pix0, const RayRec* __restrict__ rays, Hit* __restrict__ hits, Counters* ctr, const uint32_t* __restrict__ work, uint32_t* __restrict__ deferOut) {
  const long long n = work ? (long long)ctr->deferTrace[w.level] : waveCount(w, ctr);
  if (w.level == 0 && !work && blockIdx.x == 0 && threadIdx.x == 0) ctr->levelCount[0] = (unsigned long long)w.n0;
  if (work && n > 0 && blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(&ctr->deferredTotal, (unsigned long long)n);
  TraceCounters tc; tc.box = 0; tc.prim = 0;
  for (long long base = (long long)blockIdx.x * blockDim.x; base < n; base += (long long)gridDim.x * blockDim.x) {
    long long i = base + threadIdx.x; bool defer = false;
    if (i < n) {
      if (work) i = work[i];
      // the ray / hit records are pure streams (read once, written once): evict-first loads and stores keep them from pushing the scene and the
      // local-memory traversal state out of L2
      RayRec r; if (rays) loadRayRec(r, rays + i); else primaryRay(S, pm, pix0, i, r);
      Hit h; hitReset(h);
      if (r.valid) {
        Ray ray = makeRay(d3(r.o[0], r.o[1], r.o[2]), d3(r.d[0], r.d[1], r.d[2]));
        const int got = closestHitT<F>(S, ray, rayTime(S, r.stream, r.ka, r.kb, r.kc, r.stream == STREAM_PIXEL ? DIM_TIME : 0xFFFFu), h, COUNT ? &tc : nullptr);
        if (F != TF_ALL && got < 0) { defer = true; hitReset(h); }
        h.pad0 = 1;            // the ray's valid flag: k_shade reads it at level 0 instead of generating the primary ray again
      }
      if (!defer) storeHit(hits + i, h);
    }
    if (F != TF_ALL) deferAppend(defer, (uint32_t)i, &ctr->deferTrace[w.level], deferOut);
  }
  if (COUNT) { warpAdd(&ctr->box, tc.box); warpAdd(&ctr->prim, tc.prim); warpAdd(&ctr->boxC, tc.box); warpAdd(&ctr->primC, tc.prim); }
}

// skydome lookup for rays that leave the scene (myScene.java:1104-1149): nearest texel, no filtering
__device__ inline D3 skyColor(const DScene& S, D3 o, D3 d) {
  const FGlobals& g = S.g; double rx = g.skyRad[0], ry = g.skyRad[1], rz = g.skyRad[2];
  double dxr = d.x / rx, dyr = d.y / ry, dzr = d.z / rz;
  double a = ((dxr) * (dxr)) + ((dyr) * (dyr)) + ((dzr) * (dzr));
  D3 pC = d3((o.x - g.skyOrigin[0]) / rx, (o.y - g.skyOrigin[1]) / ry, (o.z - g.skyOrigin[2]) / rz);
  double b = 2 * (((dxr) * pC.x) + ((dyr) * pC.y) + ((dzr) * pC.z)), c = (pC.x * pC.x) + (pC.y * pC.y) + (pC.z * pC.z) - 1;
  double discr = ((b * b) - (4 * a * c)), t = -DRT_DMAX;
  if (discr > 0) { double d1 = sqrt(discr), t1 = (-1 * b + d1) / (2 * a), t2 = (-1 * b - d1) / (2 * a), tv = jminD(t1, t2); if (tv < DRT_EPS) tv = jmaxD(t1, t2); t = tv; }
  D3 p = d3((d.x * t) + o.x, (d.y * t) + o.y, (d.z * t) + o.z);
  const FImage im = S.images[g.skyImage];
  double a0 = p.y - g.skyOrigin[1], a1 = a0 / ry; a1 = (a1 > 1) ? 1 : (a1 < -1) ? -1 : a1;
  double v = (im.h - 1) * acos(a1) / DRT_PI;
  double shWm1 = im.w - 1, z1 = (p.z - g.skyOrigin[2]), q = v / (im.h - 1);
  double b0 = (p.x - g.skyOrigin[0]) / rx; b0 = (b0 > 1) ? 1 : (b0 < -1) ? -1 : b0;
  double b1 = sin(q * DRT_PI), b2 = (fabs(b1) < DRT_EPS) ? 1 : b0 / b1;
  double u = (z1 <= DRT_EPS) ? ((shWm1 * (acos(b2)) / (DRT_TWO_PI_F)) + shWm1 / 2.0f) : shWm1 - ((shWm1 * (acos(b2)) / (DRT_TWO_PI_F)) + shWm1 / 2.0f);
  u = (u < 0) ? 0 : (u > shWm1) ? shWm1 : u;
  long long idx = (long long)j2iD(v) * im.w + j2iD(u), n = (long long)im.w * im.h; idx = idx < 0 ? 0 : (idx >= n ? n - 1 : idx);
  return colorOfArgb(S.texels[im.offset + idx]);
}

// Surface pass. One thread per ray of the level; children go to the next level's queue (its length lives on the device: levelCount[level+1]).
// PRIMARY (level 0, rays == null): the ray's keys are functions of the index, its valid flag is in the hit record (Hit::pad0), origin and
// direction are only needed for a skydome lookup (a hit uses h.rawDir); the node record is written whole (no k_raygen pass).  One instance per
// case, so that the bounce levels carry none of the primary-ray code in their register allocation.
#ifndef DRT_SHADE_MINBLOCKS
#define DRT_SHADE_MINBLOCKS 4
#endif
template <bool PRIMARY>
__global__ void __launch_bounds__(128, DRT_SHADE_MINBLOCKS) k_shade(const __grid_constant__ DScene S, Wave w, PixMap pm, long long pix0, const RayRec* __restrict__ rays, const Hit* __restrict__ hits,
                                               SurfRec* __restrict__ surf, NodeRec* __restrict__ nodesBase, RayRec* __restrict__ nextRays, Counters* ctr) {
  const long long n = waveCount(w, ctr);
  const long long off = PRIMARY ? 0 : waveNodeOffset(w, ctr, w.level), offNext = off + n;
  NodeRec* __restrict__ nodes = nodesBase + off; NodeRec* __restrict__ nextNodes = nodesBase + offNext;
  const long long nextCap = (w.nodeCap - offNext) < w.rayCap ? (w.nodeCap - offNext) : w.rayCap;
  const unsigned lane = threadIdx.x & 31;
  unsigned long long cntPrimary = 0, cntRefl = 0, cntRefr = 0;
  for (long long base = (long long)blockIdx.x * blockDim.x; base < n; base += (long long)gridDim.x * blockDim.x) {
  const long long i = base + threadIdx.x;
  // up to two children per hit: A = refraction (slot 1), B = reflection (slot 2). Kept in named registers (no dynamically indexed local arrays)
  bool hasA = false, hasB = false; D3 dirA = d3(0, 0, 0), wA = dirA, dirB = dirA, wB = dirA, orgC = dirA; double ktA0 = 1, ktA1 = 1, ktB0 = 1, ktB1 = 1;
  uint32_t cka = 0, ckb = 0, ckc = 0, cstream = 0; int32_t cgen = 0;
  bool cPrimary = false, cRefl = false, cRefr = false;
  if (i < n) {
    const Hit h = hits[i];
    RayRec r;
    if constexpr (!PRIMARY) r = rays[i];
    else if (S.g.hasSky && h.prim < 0) primaryRay(S, pm, pix0, i, r);
    else { const PixKey k = pixelOf(S.g, pm, pix0, i); r.ka = (uint32_t)k.pix; r.kb = k.smp; r.kc = 1; r.stream = STREAM_PIXEL; r.gen = 0; r.valid = h.pad0; r.kt0 = 1; r.kt1 = 1; }
    SurfRec s; s.valid = 0; s.shader = -1; s.ka = r.ka; s.kb = r.kb; s.kc = r.kc; s.stream = r.stream; s.gen = r.gen; s.pad = 0;
    D3 local = d3(0, 0, 0);
    if (r.valid) {
      if (r.gen == 0) cPrimary = true;
      if (h.prim < 0) {
        if (S.g.hasSky) local = skyColor(S, d3(r.o[0], r.o[1], r.o[2]), d3(r.d[0], r.d[1], r.d[2]));
        else local = d3(S.g.bg[0], S.g.bg[1], S.g.bg[2]);
      } else {
        const FPrim P = S.prims[h.prim]; const FXform& X = S.xforms[h.hitXform];
        const int shIdx = h.shaderOverride >= 0 ? h.shaderOverride : P.shader; const FShader sh = S.shaders[shIdx];
        D3 fwd = xfPoint(X.m, h.loc);
        D3 nrm = norm3(xfVector(X.adj, primNormal(S, P, h.loc, h.arg0, h.arg1, h.state)));
        local = d3(sh.amb[0], sh.amb[1], sh.amb[2]);
        const bool simple = (sh.flags & SF_SIMPLE) != 0;       // (the photon term is added by k_photon_gather, which runs next)
        double time = rayTime(S, r.stream, r.ka, r.kb, r.kc, DIM_TIME);
        D3 tex = evalTexture(S, sh, P, h.loc, fwd, h.state, time);
        s.valid = 1; s.shader = shIdx;
        s.loc[0] = fwd.x; s.loc[1] = fwd.y; s.loc[2] = fwd.z; s.n[0] = nrm.x; s.n[1] = nrm.y; s.n[2] = nrm.z;
        s.rawDir[0] = h.rawDir.x; s.rawDir[1] = h.rawDir.y; s.rawDir[2] = h.rawDir.z; s.tex[0] = tex.x; s.tex[1] = tex.y; s.tex[2] = tex.z;
        // secondary rays (leave room for the shadow generation: gen < numRays - 2)
        if ((r.gen < S.g.numRays - 2) && (sh.flags & SF_HAS_CAUSTIC)) {
          orgC = fwd; cka = r.ka; ckb = r.kb; ckc = r.kc; cstream = r.stream; cgen = r.gen + 1;
          auto child = [&](int slot, D3 dir, D3 wgt, double kt0, double kt1) {
            if (slot == 1) { hasA = true; dirA = norm3(dir); wA = wgt; ktA0 = kt0; ktA1 = kt1; } else { hasB = true; dirB = norm3(dir); wB = wgt; ktB0 = kt0; ktB1 = kt1; }
          };
          D3 perm = d3(sh.perm[0], sh.perm[1], sh.perm[2]);
          bool trans = simple ? (sh.KTrans > 0) : ((sh.KTrans > 0) || (sh.currPerm > 0.0));
          if (trans) {
            Fres f = simple ? fresnel(h.rawDir, nrm, sh.currPerm, r.kt1) : fresnel(h.rawDir, nrm, sh.KTrans, r.kt0);
            const double thr = simple ? 0.0 : DRT_EPS;
            if (f.oneM > thr) { D3 wgt = simple ? d3(f.oneM * sh.KTrans, f.oneM * sh.KTrans, f.oneM * sh.KTrans) : d3((f.oneM) * perm.x, (f.oneM) * perm.y, (f.oneM) * perm.z);
              child(1, refractDir(f), wgt, sh.KTrans, sh.currPerm); cRefr = true; }
            if (f.ratio > thr) { D3 rd = scale3(reflDir(f.back, f.N), f.mult);
              D3 wgt = simple ? d3(f.ratio * sh.KRefl, f.ratio * sh.KRefl, f.ratio * sh.KRefl) : d3((f.ratio) * perm.x, (f.ratio) * perm.y, (f.ratio) * perm.z);
              if (simple) child(2, rd, wgt, 1, 1); else child(2, rd, wgt, sh.KTrans, sh.currPerm); cRefl = true; }
          } else if (sh.KRefl > 0.0) {
            D3 back = scale3(h.rawDir, -1); D3 rd = reflDir(back, nrm);
            if (dot3(rd, nrm) >= 0) { child(2, rd, d3(sh.kreflClr[0], sh.kreflClr[1], sh.kreflClr[2]), 1, 1); cRefl = true; }
          }
        }
      }
    }
    surf[i] = s;
    if constexpr (!PRIMARY) { nodes[i].local[0] = local.x; nodes[i].local[1] = local.y; nodes[i].local[2] = local.z; }
    else { NodeRec nd; nd.parent = -1; nd.slot = 0; nd.pad[0] = nd.pad[1] = 0; nd.local[0] = local.x; nd.local[1] = local.y; nd.local[2] = local.z;
      for (int k = 0; k < 3; ++k) { nd.cA[k] = 0; nd.cB[k] = 0; nd.w[k] = 1; } nodes[i] = nd; }
  }
  // warp-aggregated compaction of the children into the next level's queue
  const int nChild = (hasA ? 1 : 0) + (hasB ? 1 : 0);
  int incl = nChild;
  for (int o = 1; o < 32; o <<= 1) { int v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= (unsigned)o) incl += v; }
  int total = __shfl_sync(0xffffffffu, incl, 31);
  unsigned long long qbase = 0;
  if (total > 0) {
    if (lane == 31) { qbase = atomicAdd(&ctr->levelCount[w.level + 1], (unsigned long long)total);
      if (ctr->maxLevel < (unsigned long long)(w.level + 1)) atomicMax(&ctr->maxLevel, (unsigned long long)(w.level + 1));
      if (w.level + 1 >= w.launchedLevels) flagError(DEV_ERR_DEPTH);                    // deeper than the levels this call launched: the host re-renders with full depth
      if ((long long)(qbase + total) > nextCap) flagError(DEV_ERR_QUEUE); }               // queue / node pool exhausted: the host re-renders with smaller batches
    qbase = __shfl_sync(0xffffffffu, qbase, 31);
  }
  long long at = (long long)qbase + (incl - nChild);
  auto emit = [&](long long pos, int slot, D3 dn, D3 wgt, double kt0, double kt1) {
    if (pos >= nextCap) return;
    RayRec c; c.o[0] = orgC.x; c.o[1] = orgC.y; c.o[2] = orgC.z; c.d[0] = dn.x; c.d[1] = dn.y; c.d[2] = dn.z; c.kt0 = kt0; c.kt1 = kt1;
    c.ka = cka; c.kb = ckb; c.kc = ckc * 2 + (slot == 1 ? 1 : 0); c.stream = cstream; c.gen = cgen; c.valid = 1; c.pad[0] = c.pad[1] = 0;
    NodeRec nn; nn.parent = (int32_t)i; nn.slot = slot; nn.pad[0] = nn.pad[1] = 0; nn.w[0] = wgt.x; nn.w[1] = wgt.y; nn.w[2] = wgt.z;
    for (int k = 0; k < 3; ++k) { nn.local[k] = 0; nn.cA[k] = 0; nn.cB[k] = 0; }
    nextRays[pos] = c; nextNodes[pos] = nn;
  };
  if (hasA) emit(at, 1, dirA, wA, ktA0, ktA1);
  if (hasB) emit(at + (hasA ? 1 : 0), 2, dirB, wB, ktB0, ktB1);
  // 0/1 flags: one ballot + popc per counter instead of a 64-bit shuffle tree
  cntPrimary += __popc(__ballot_sync(0xffffffffu, cPrimary)); cntRefl += __popc(__ballot_sync(0xffffffffu, cRefl)); cntRefr += __popc(__ballot_sync(0xffffffffu, cRefr));
  }
  if (lane == 0) { if (cntPrimary) atomicAdd(&ctr->primaryS[blockIdx.x & 63], cntPrimary); if (cntRefl) atomicAdd(&ctr->reflect, cntRefl); if (cntRefr) atomicAdd(&ctr->refract, cntRefr); }
}

// Light pass: literal calcShadowColor, one thread per shaded hit, lights in list order, shadow rays traced in-thread.
// F / work / deferOut as in k_trace: a lean variant that meets a shadow ray it cannot serve leaves the WHOLE record to the generic pass
// (the record's light sum is formed by one thread in list order either way).
// Register budget: only what the shadow ray needs (hit point, keys, running sum) is held across the BVH walk; the normal, texture colour,
// ray direction and shader / light constants of the shading that follows are read from the (L1/L2-resident) records after the walk.  Held
// across it at the 80-register cap, they were spilled to local memory and written back through L2 on every light.
__device__ __forceinline__ D3 ldgD3(const double* p) { return d3(__ldg(p), __ldg(p + 1), __ldg(p + 2)); }
template <bool COUNT, int F>
__global__ void __launch_bounds__(128, lightMinBlocks(F))
k_light(const __grid_constant__ DScene S, Wave w, const SurfRec* __restrict__ surf, NodeRec* __restrict__ nodesBase, Counters* ctr, const uint32_t* __restrict__ work, uint32_t* __restrict__ deferOut) {
  const long long n = work ? (long long)ctr->deferLight[w.level] : waveCount(w, ctr);
  NodeRec* __restrict__ nodes = nodesBase + ((w.level == 0) ? 0 : waveNodeOffset(w, ctr, w.level));
  if (work && n > 0 && blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(&ctr->deferredTotal, (unsigned long long)n);
  TraceCounters tc; tc.box = 0; tc.prim = 0; unsigned long long cShadow = 0;
  for (long long base = (long long)blockIdx.x * blockDim.x; base < n; base += (long long)gridDim.x * blockDim.x) {
    long long i = base + threadIdx.x; bool defer = false;
    if (i < n) {
      if (work) i = work[i];
      const SurfRec* __restrict__ s = surf + i;
      const int4 sv = __ldg(reinterpret_cast<const int4*>(&s->shader));            // shader, valid, ka, kb
      if (sv.y) {
        const int2 sk = __ldg(reinterpret_cast<const int2*>(&s->kc));               // kc, stream
        const uint32_t ka = (uint32_t)sv.z, kb = (uint32_t)sv.w, kc = (uint32_t)sk.x, stream = (uint32_t)sk.y;
        const FShader& sh = S.shaders[sv.x];
        const D3 hitLoc = ldgD3(s->loc);
        double r = 0, g = 0, b = 0; unsigned nShadow = 0;
        for (int li = 0; li < S.g.numLights; ++li) {
          const FLight& L = S.lights[li];
          const uint32_t dim = DIM_LIGHT_BASE + DIM_LIGHT_STRIDE * li;
          const int type = L.type;
          D3 lo = d3(L.origin[0], L.origin[1], L.origin[2]), orient = d3(L.orient[0], L.orient[1], L.orient[2]);
          auto diskPos = [&](uint32_t d0) {           // myDiskLight.getRandomDiskPos (:251-258)
            double ua = philoxU01(S.g.seed, stream, ka, kb, kc, d0), ur = philoxU01(S.g.seed, stream, ka, kb, kc, d0 + 1);
            D3 tmp = norm3(rotAboutAxis(d3(L.tangent[0], L.tangent[1], L.tangent[2]), orient, urange(ua, 0, DRT_TWO_PI_F)));
            return add3(scale3(tmp, urange(ur, 0, L.radius)), lo);
          };
          // world position of the sample on the light: per ray for a disk, else the light's transformed origin (S.lightPos, formed once per upload)
          const D3 target = (type == LT_DISK) ? xfPoint(S.xforms[L.xform].m, diskPos(dim)) : ldgD3(S.lightPos + 3 * li);
          D3 lightNorm = norm3(sub3(target, hitLoc));
          Ray shadowRay = makeRay(hitLoc, lightNorm);
          // light.intersectCheck: distance to the light's (re-sampled, untransformed) origin, penumbra factor (SURVEY Q12)
          D3 dOrg = (type == LT_DISK) ? diskPos(dim + 2) : lo;
          double t = sqrt(((hitLoc.x - dOrg.x) * (hitLoc.x - dOrg.x)) + ((hitLoc.y - dOrg.y) * (hitLoc.y - dOrg.y)) + ((hitLoc.z - dOrg.z) * (hitLoc.z - dOrg.z)));
          double ltMult = 1;
          if (type == LT_SPOT) { double angle = acos(-1 * dot3(lightNorm, orient)); ltMult = (angle < L.innerRad) ? 1 : (angle > L.outerRad) ? 0 : (L.outerRad - angle) / L.radDiff; }
          if (ltMult == 0) continue;
          ++nShadow;
          double time = rayTime(S, stream, ka, kb, kc, dim + 4);
          const int occluded = anyHitT<F>(S, shadowRay, time, t, COUNT ? &tc : nullptr);
          if (F != TF_ALL && occluded < 0) { defer = true; break; }
          if (!occluded) {
            const D3 N = ldgD3(s->n), tex = ldgD3(s->tex), color = d3(L.color[0], L.color[1], L.color[2]);
            double ld = dot3(lightNorm, N) * ltMult;
            if (ld > DRT_EPS) { r += tex.x * color.x * ld; g += tex.y * color.y * ld; b += tex.z * color.z * ld; }
            const double phong = sh.phong;
            if (phong == 0) continue;
            D3 hN = norm3(sub3(lightNorm, ldgD3(s->rawDir)));
            double hd = dot3(hN, N) * ltMult;
            if (hd > DRT_EPS) { double ph = pow(hd * hd, phong); r += sh.spec[0] * color.x * ph; g += sh.spec[1] * color.y * ph; b += sh.spec[2] * color.z * ph; }
          }
        }
        if (!defer) { cShadow += nShadow; nodes[i].local[0] += r; nodes[i].local[1] += g; nodes[i].local[2] += b; }
      }
    }
    if (F != TF_ALL) deferAppend(defer, (uint32_t)i, &ctr->deferLight[w.level], deferOut);
  }
  warpAdd(&ctr->shadowS[blockIdx.x & 63], cShadow);
  if (COUNT) { warpAdd(&ctr->box, tc.box); warpAdd(&ctr->prim, tc.prim); }
}
// world position of every light's origin, xfPoint(CTM, origin): the target of every shadow ray toward a point or spot light
__global__ void k_light_pos(const FXform* __restrict__ xforms, const FLight* __restrict__ lights, int n, double* __restrict__ out) {
  const int li = blockIdx.x * blockDim.x + threadIdx.x; if (li >= n) return;
  const FLight L = lights[li]; const D3 p = xfPoint(xforms[L.xform].m, d3(L.origin[0], L.origin[1], L.origin[2]));
  out[3 * li] = p.x; out[3 * li + 1] = p.y; out[3 * li + 2] = p.z;
}

__device__ __forceinline__ D3 nodeTotal(const NodeRec& nd) {
  return clampColor1(d3(nd.local[0] + (nd.cA[0] + nd.cB[0]), nd.local[1] + (nd.cA[1] + nd.cB[1]), nd.local[2] + (nd.cA[2] + nd.cB[2])));
}
// level L -> level L-1: parent.slot = w (.) clamp1(total(child)).  The level's length and position are read from the device counters.
__global__ void k_resolve(Wave w, NodeRec* __restrict__ nodesBase, const Counters* ctr) {
  const long long n = waveCount(w, ctr), off = waveNodeOffset(w, ctr, w.level), offP = waveNodeOffset(w, ctr, w.level - 1);
  const NodeRec* __restrict__ lvl = nodesBase + off; NodeRec* __restrict__ parentLvl = nodesBase + offP;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const NodeRec nd = lvl[i]; D3 c = nodeTotal(nd);
    double* dst = (nd.slot == 1) ? parentLvl[nd.parent].cA : parentLvl[nd.parent].cB;
    dst[0] = nd.w[0] * c.x; dst[1] = nd.w[1] * c.y; dst[2] = nd.w[2] * c.z;
  }
}
__global__ void k_finish(const __grid_constant__ DScene S, PixMap pm, long long pix0, long long nPix, const NodeRec* __restrict__ roots, const Hit* __restrict__ hits0, RenderOutputs out) {
  long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; if (p >= nPix) return;
  long long q = absPixel(pm, pix0 + p); if (q >= pm.totalPix) return;
  int spp = S.g.spp < 1 ? 1 : S.g.spp; double r = 0, g = 0, b = 0;
  for (int s = 0; s < spp; ++s) { D3 c = nodeTotal(roots[p * spp + s]); r += c.x; g += c.y; b += c.z; }
  D3 c;
  if (S.g.spp < 1) c = d3(0, 0, 0);
  else c = clampColor1(d3(r / spp, g / spp, b / spp));
  if (out.argb) out.argb[out.packed ? (pix0 + p) : q] = packArgb(c);
  if (out.rgb) { out.rgb[3 * q] = c.x; out.rgb[3 * q + 1] = c.y; out.rgb[3 * q + 2] = c.z; }
  if (out.hitPrim || out.hitInst || out.t) {
    const Hit h = hits0[p * spp];
    if (out.hitPrim) out.hitPrim[q] = h.prim >= 0 ? S.prims[h.prim].serial : -1;
    if (out.hitInst) out.hitInst[q] = h.prim >= 0 ? h.inst : -1;
    if (out.t) out.t[q] = h.prim >= 0 ? h.t : 0;
  }
}

// FP32 mirror of GPU-built nodes (DRT_ACCEL_LBVH); host-built nodes are mirrored by the flattener
__global__ void k_nodes32(const FNode* __restrict__ in, long long n, FNode32* __restrict__ out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; if (i >= n) return;
  const FNode a = in[i]; FNode32 m;
  for (int k = 0; k < 3; ++k) { m.lmin[k] = (float)a.lmin[k]; m.lmax[k] = (float)a.lmax[k]; m.rmin[k] = (float)a.rmin[k]; m.rmax[k] = (float)a.rmax[k]; }
  m.left = a.left; m.right = a.right; m.triL = a.triL; m.triR = a.triR; out[i] = m;
}

// caller ray queries (drt_query_closest / drt_query_occluded) -----------------------------------------------------
// One thread = one caller ray (FP64 origin and direction, 3 doubles each, ray time 0), through rayLoop: the scene's lean variant defers what
// it cannot serve to `deferOut` (count in Counters::deferTrace[0] / deferLight[0]), the generic variant serves everything and is the fix-up
// pass over that list.  A ray is traced only if origin and direction are finite and the direction's FP64 length is finite and nonzero; any
// other ray is a miss / not occluded.
__device__ __forceinline__ bool queryRay(const double* __restrict__ org, const double* __restrict__ dir, long long i, Ray& ray) {
  const D3 o = d3(org[3 * i], org[3 * i + 1], org[3 * i + 2]), d = d3(dir[3 * i], dir[3 * i + 1], dir[3 * i + 2]);
  const double m = mag3(d);
  if (!(isfinite(o.x) && isfinite(o.y) && isfinite(o.z) && isfinite(d.x) && isfinite(d.y) && isfinite(d.z) && isfinite(m) && m > 0)) return false;
  ray = makeRay(o, norm3(d)); return true;
}
// closest hit, reported as a miss unless t < tmax[i] (tmax == null: +inf).  The search itself is the unbounded one.  pos / nrm (optional): the
// world hit point and unit normal k_shade shades with (0 on a miss).  k_query_closest<TF_ALL> is also the drt_trace_rays probe.
template <int F>
__global__ void __launch_bounds__(128, traceMinBlocks(F))
k_query_closest(const __grid_constant__ DScene S, long long nRays, const double* __restrict__ org, const double* __restrict__ dir, const double* __restrict__ tmax,
                int32_t* __restrict__ ids, double* __restrict__ tOut, double* __restrict__ pos, double* __restrict__ nrm, Counters* ctr, const uint32_t* __restrict__ work, uint32_t* __restrict__ deferOut) {
  rayLoop<F>(nRays, work, &ctr->deferTrace[0], deferOut, ctr, [&](long long i) __attribute__((always_inline)) {
    Hit h; hitReset(h); Ray ray; bool defer = false;
    if (queryRay(org, dir, i, ray)) {
      const int got = closestHitT<F>(S, ray, 0.0, h, nullptr);
      if (F != TF_ALL && got < 0) defer = true;
    }
    if (!defer) {
      const bool hit = h.prim >= 0 && (!tmax || h.t < tmax[i]);
      ids[2 * i] = hit ? S.prims[h.prim].serial : -1; ids[2 * i + 1] = hit ? h.inst : -1; tOut[i] = hit ? h.t : 0;
      if (pos || nrm) {
        D3 p = d3(0, 0, 0), q = p;
        if (hit) {
          const FPrim P = S.prims[h.prim]; const FXform& X = S.xforms[h.hitXform];
          p = xfPoint(X.m, h.loc); q = norm3(xfVector(X.adj, primNormal(S, P, h.loc, h.arg0, h.arg1, h.state)));
        }
        if (pos) { pos[3 * i] = p.x; pos[3 * i + 1] = p.y; pos[3 * i + 2] = p.z; }
        if (nrm) { nrm[3 * i] = q.x; nrm[3 * i + 1] = q.y; nrm[3 * i + 2] = q.z; }
      }
    }
    return defer;
  });
}
// occlusion: the renderer's shadow test (anyHitT: something hit with (dist - t) > DRT_EPS).  dist may be +inf; a NaN dist is not occluded
template <int F>
__global__ void __launch_bounds__(128, lightMinBlocks(F))
k_query_any(const __grid_constant__ DScene S, long long nRays, const double* __restrict__ org, const double* __restrict__ dir, const double* __restrict__ dist,
            uint8_t* __restrict__ occluded, Counters* ctr, const uint32_t* __restrict__ work, uint32_t* __restrict__ deferOut) {
  rayLoop<F>(nRays, work, &ctr->deferLight[0], deferOut, ctr, [&](long long i) __attribute__((always_inline)) {
    const double d = dist[i]; int got = 0; Ray ray; bool defer = false;
    if (d == d && queryRay(org, dir, i, ray)) {
      got = anyHitT<F>(S, ray, 0.0, d, nullptr);
      if (F != TF_ALL && got < 0) defer = true;
    }
    if (!defer) occluded[i] = got > 0 ? 1 : 0;
    return defer;
  });
}

// parity helper ------------------------------------------------------------------------------------------------
__global__ void k_eval_texture(const __grid_constant__ DScene S, int shader, long long n, const double* __restrict__ hl, const double* __restrict__ fl, double* __restrict__ out) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; if (i >= n) return;
  FPrim P; P.type = PT_BOX; P.flags = 0; P.xform = 0; P.shader = shader; P.data = 0; P.serial = 0; P.pad0 = P.pad1 = 0;   // no image textures through this probe
  D3 c = evalTexture(S, S.shaders[shader], P, d3(hl[3 * i], hl[3 * i + 1], hl[3 * i + 2]), d3(fl[3 * i], fl[3 * i + 1], fl[3 * i + 2]), 0, 0.0);
  out[3 * i] = c.x; out[3 * i + 1] = c.y; out[3 * i + 2] = c.z;
}

}  // namespace drt

#include "photon.cuh"
#include "lbvh.cuh"
#include "refbvh.cuh"

namespace drt {

// ---------------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------------
// Scene arrays live in ONE device arena fed from ONE pinned host staging buffer (grow-only): a re-upload is a host memcpy per array plus a
// single H2D DMA -- no cudaMalloc / cudaFree on the per-frame path.
struct SceneArena {
  char* dev = nullptr; char* host = nullptr; size_t cap = 0, used = 0;
  SceneArena() = default;
  SceneArena(const SceneArena&) = delete; SceneArena& operator=(const SceneArena&) = delete;
  ~SceneArena() { if (dev) cudaFree(dev); if (host) cudaFreeHost(host); }
  void reserve(size_t bytes, cudaStream_t st) {
    if (bytes <= cap) return;
    CK(cudaStreamSynchronize(st)); if (dev) cudaFree(dev); if (host) cudaFreeHost(host);
    cap = bytes + bytes / 4 + (1 << 20); CK(cudaMalloc(&dev, cap)); CK(cudaMallocHost(&host, cap)); stagedScene = nullptr;
  }
  bool fill = true;                      // false: the staging buffer already holds exactly this scene (a re-upload): only the DMA is repeated
  const void* stagedScene = nullptr; size_t stagedUsed = 0;
  void begin() { used = 0; }
  template <class T> const T* put(const std::vector<T>& v) {
    used = (used + 255) & ~(size_t)255; const size_t at = used; const size_t n = v.size() * sizeof(T);
    if (fill && n) std::memcpy(host + at, v.data(), n);
    used += n ? n : sizeof(T); return reinterpret_cast<const T*>(dev + at);
  }
  template <class T> static size_t need(const std::vector<T>& v) { return ((v.size() ? v.size() : 1) * sizeof(T) + 255) & ~(size_t)255; }
  void flush(cudaStream_t st) { if (used) CK(cudaMemcpyAsync(dev, host, used, cudaMemcpyHostToDevice, st)); }
};

// Everything the renderer allocates on its device; created with that device current, freed with the renderer.
struct Renderer::Impl {
  DScene ds; SceneArena arena; DBuf<FNode> lbvhNodeBuf; DBuf<FNode32> lbvhNode32Buf; DBuf<FTri> lbvhTriBuf; LbvhScratch lbvhScratch; RefBvhScratch refScratch;
  DBuf<RayRec> rays[2]; DBuf<Hit> hits; DBuf<Hit> hits0; DBuf<SurfRec> surf; DBuf<NodeRec> nodes; DBuf<double> lightPos; Counters* ctr = nullptr; Counters* ctrHost = nullptr;
  DBuf<uint32_t> deferT, deferL;                 // deferral lists of the lean trace / light kernels (ray indices of one level)
  std::vector<DEvent> evPool;                    // stage timing of a whole frame without a host sync per level
  int shape = TF_ALL;                            // kernel variant the uploaded scene runs with (see chooseShape)
  // the lean kernel of a pass for `shape`, given its F = 0 and F = TF_LITERAL1 instances; null when only the generic kernel serves the scene
  template <class K> K lean(K shape0, K literal1) const { return shape == TF_ALL ? nullptr : shape == 0 ? shape0 : literal1; }
  bool anySecondary = false;                     // some shader can spawn reflection / refraction rays
  int depthHint = 0;                             // levels the last frame of this scene needed (0 = unknown: launch the full depth)
  double capHint = 0;                            // queue-capacity factor the last frame of this scene ended up with (0 = default)
  int numSMs = 148;
  cudaEvent_t pev(size_t k) { while (evPool.size() <= k) evPool.emplace_back(); return evPool[k]; }
  DBuf<int32_t> oArgb, oPrim, oInst; DBuf<double> oRgb, oT;
  DBuf<double> probeIn[2], probeOut[2];          // inputs and outputs of the parity probes
  DEvent lbvhEv[2];
  PhotonMap photons; DBuf<unsigned long long> xCnt; DBuf<PhotonRec> xMine, xAll;      // photon record exchange of drt_render_distributed
  size_t sceneBytes = 0;
  float lbvhMs = 0; long long lbvhTris = 0, lbvhNodes = 0;
  std::vector<FBvh> bvhsUploaded;                // host copy of the FBvh array as uploaded (fastRoot points at the LBVH nodes in DRT_ACCEL_LBVH mode)
  Impl() { CK(cudaMalloc(&ctr, sizeof(Counters))); CK(cudaMallocHost(&ctrHost, sizeof(Counters))); }
  ~Impl() { cudaFree(ctr); cudaFreeHost(ctrHost); }
};

Renderer::Renderer(int device) : device_(device) {
  int cnt = 0; cudaError_t e = cudaGetDeviceCount(&cnt);
  if (e != cudaSuccess || cnt == 0) throw std::runtime_error("no CUDA device available: this renderer has no CPU fallback");
  CK(cudaSetDevice(device));
  impl_.reset(new Impl);
  { cudaDeviceProp pr; CK(cudaGetDeviceProperties(&pr, device)); impl_->numSMs = pr.multiProcessorCount; }
  std::memset(&impl_->ds, 0, sizeof(DScene)); std::memset(&g_, 0, sizeof(g_));
  static const unsigned char p[256] = {151,160,137,91,90,15,131,13,201,95,96,53,194,233,7,225,140,36,103,30,69,142,8,99,37,240,21,10,23,190,6,148,247,120,234,75,0,26,197,62,94,252,219,203,117,35,11,32,57,177,33,88,237,149,56,87,174,20,125,136,171,168,68,175,74,165,71,134,139,48,27,166,77,146,158,231,83,111,229,122,60,211,133,230,220,105,92,41,55,46,245,40,244,102,143,54,65,25,63,161,1,216,80,73,209,76,132,187,208,89,18,169,200,196,135,130,116,188,159,86,164,100,109,198,173,186,3,64,52,217,226,250,124,123,5,202,38,147,118,126,255,82,85,212,207,206,59,227,47,16,58,17,182,189,28,42,223,183,170,213,119,248,152,2,44,154,163,70,221,153,101,155,167,43,172,9,129,22,39,253,19,98,108,110,79,113,224,232,178,185,112,104,218,246,97,228,251,34,242,193,238,210,144,12,191,179,162,241,81,51,145,235,249,14,239,107,49,192,214,31,181,199,106,157,184,84,204,176,115,121,50,45,127,4,150,254,138,236,205,93,222,114,67,29,24,72,243,141,128,195,78,66,215,61,156,180};
  unsigned char perm[512]; for (int i = 0; i < 512; ++i) perm[i] = p[i & 255];
  CK(cudaMemcpyToSymbol(c_perm, perm, 512));
  cudaStream_t st; CK(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking)); stream_ = st;
}
// impl_ is destroyed after the body, with the device still current
Renderer::~Renderer() { cudaSetDevice(device_); commDestroy(); cudaStreamDestroy((cudaStream_t)stream_); }

// object order of the reference-topology median-split tree on the device (refbvh.cuh); false = the host recursion has to do it
bool Renderer::orderBvh(int n, const double* keys, int32_t* ord, double* ms) {
  CK(cudaSetDevice(device_));
  return refOrderDevice(n, keys, ord, impl_->refScratch, (cudaStream_t)stream_, ms);
}

void Renderer::upload(const HostScene& hs, bool sameScene) {
  keepDepthHint_ = sameScene;
  CK(cudaSetDevice(device_)); cudaStream_t st = (cudaStream_t)stream_;
  CK(cudaStreamSynchronize(st));
  // device-side nesting limits (see dev_isect.cuh): accel children are primitives or instances; an instanced accel holds primitives
  std::vector<char> seenBase[2] = {std::vector<char>(hs.lists.size(), 0), std::vector<char>(hs.bvhs.size(), 0)};      // 21 845 instances of one mesh: check the mesh once
  for (const FInstance& in : hs.instances) if (in.baseKind == OK_LIST || in.baseKind == OK_BVH) {
    { std::vector<char>& seen = seenBase[in.baseKind == OK_BVH ? 1 : 0]; if (in.baseIdx >= 0 && (size_t)in.baseIdx < seen.size()) { if (seen[in.baseIdx]) continue; seen[in.baseIdx] = 1; } }
    auto checkList = [&](const FList& L) { for (int i = 0; i < L.childCount; ++i) { const FObjRef& c = hs.children[L.childStart + i];
      if (c.kind == OK_INSTANCE && hs.instances[c.idx].baseKind != OK_PRIM) throw std::runtime_error("instances nested deeper than TLAS->instance->BLAS are not supported on the device"); } };
    if (in.baseKind == OK_LIST) checkList(hs.lists[in.baseIdx]);
    else { std::vector<int32_t> st2{hs.bvhs[in.baseIdx].root}; while (!st2.empty()) { int32_t r = st2.back(); st2.pop_back(); if (r < 0) checkList(hs.lists[~r]); else { st2.push_back(hs.nodes[r].left); st2.push_back(hs.nodes[r].right); } } }
  }
  DScene& d = impl_->ds; SceneArena& A = impl_->arena;
  std::vector<FBvh> bv = hs.bvhs;
  d.accelMode = accelMode_; d.padA = 0;
  // DRT_ACCEL_LBVH: every qualifying pure-triangle BVH is rebuilt on the GPU (lbvh.cuh) after the copy. Node slots: the reference nodes
  // first (instance-level trees, BVHs that do not qualify, rays whose units forbid reordering keep using them), LBVH nodes appended.
  size_t extra = 0;
  if (d.accelMode == 2) for (FBvh& B : bv) if (B.fast && B.triXform == B.xform && B.triCount > 4) { B.fastRoot = (int32_t)(hs.nodes.size() + extra); extra += (size_t)((B.triCount + 3) / 4 - 1);
    // LBVH node boxes are unions of the triangles' own boxes padded by 1e-12: bound them by the vertices
    for (int k = 0; k < 3; ++k) { double m = 0; for (int t = B.triStart; t < B.triStart + B.triCount; ++t) for (int v = 0; v < 3; ++v) m = std::max(m, std::fabs(hs.tris[t].v[3 * v + k]));
      B.absMax[k] = (float)(m * (1.0 + 1e-6) + 1e-9); } }
  A.reserve(SceneArena::need(hs.xforms) + SceneArena::need(hs.prims) + SceneArena::need(hs.pdata) + SceneArena::need(hs.top) + SceneArena::need(hs.children) + SceneArena::need(hs.instances) +
            SceneArena::need(hs.lists) + SceneArena::need(hs.nodes) + SceneArena::need(hs.nodes32) + SceneArena::need(hs.tris) + SceneArena::need(bv) + SceneArena::need(hs.lights) + SceneArena::need(hs.shaders) +
            SceneArena::need(hs.textures) + SceneArena::need(hs.texColors) + SceneArena::need(hs.images) + SceneArena::need(hs.texels) + 4096, st);
  // drt_scene_reupload of the scene that is already staged: the pinned buffer still holds it byte for byte, so the host-side copies are skipped
  // and only the H2D DMA is repeated (e2e timing: "host -> device copy of the step's inputs from pinned host memory")
  const size_t needBytes = SceneArena::need(hs.xforms) + SceneArena::need(hs.prims) + SceneArena::need(hs.pdata) + SceneArena::need(hs.children) + SceneArena::need(hs.nodes) + SceneArena::need(hs.tris) + SceneArena::need(hs.texels);
  A.fill = !(sameScene && A.stagedScene == (const void*)&hs && A.stagedUsed == needBytes);
  A.begin();
  d.xforms = A.put(hs.xforms); d.prims = A.put(hs.prims); d.pdata = A.put(hs.pdata); d.top = A.put(hs.top); d.children = A.put(hs.children); d.instances = A.put(hs.instances);
  d.lists = A.put(hs.lists); d.nodes = A.put(hs.nodes); d.fnodes32 = A.put(hs.nodes32); d.tris = A.put(hs.tris); d.bvhs = A.put(bv); d.lights = A.put(hs.lights); d.shaders = A.put(hs.shaders);
  d.textures = A.put(hs.textures); d.texColors = A.put(hs.texColors); d.images = A.put(hs.images); d.texels = A.put(hs.texels);
  A.flush(st); A.stagedScene = (const void*)&hs; A.stagedUsed = needBytes; A.fill = true;
  { const int nl = (int)hs.lights.size(); impl_->lightPos.ensure(3 * (size_t)std::max(nl, 1), st); d.lightPos = impl_->lightPos.p;
    if (nl) { k_light_pos<<<(unsigned)((nl + 127) / 128), 128, 0, st>>>(d.xforms, d.lights, nl, impl_->lightPos.p); ++g_kernelLaunches; CK(cudaGetLastError()); } }
  d.fnodes = d.nodes; impl_->lbvhMs = 0; impl_->lbvhTris = 0; impl_->lbvhNodes = 0; impl_->bvhsUploaded = bv;
  if (extra) {
    const size_t n0 = hs.nodes.size();
    impl_->lbvhNodeBuf.ensure(n0 + extra, st); impl_->lbvhTriBuf.ensure(hs.tris.size(), st);
    FNode* ln = impl_->lbvhNodeBuf.p; FTri* lt = impl_->lbvhTriBuf.p;
    if (n0) CK(cudaMemcpyAsync(ln, d.nodes, n0 * sizeof(FNode), cudaMemcpyDeviceToDevice, st));
    CK(cudaMemcpyAsync(lt, d.tris, hs.tris.size() * sizeof(FTri), cudaMemcpyDeviceToDevice, st));
    { size_t mx = 0; for (const FBvh& B : bv) if (B.fast && B.fastRoot != B.root) mx = std::max(mx, (size_t)B.triCount); impl_->lbvhScratch.ensure(mx, st); }   // scratch is grow-only and allocated outside the timed build
    CK(cudaEventRecord(impl_->lbvhEv[0], st));
    for (const FBvh& B : bv) if (B.fast && B.fastRoot != B.root) {
      const int wrote = lbvhBuild(lt, B.triStart, B.triCount, B.bmin, B.bmax, ln + B.fastRoot, B.fastRoot, impl_->lbvhScratch, st);
      if (wrote != (B.triCount + 3) / 4 - 1) throw std::runtime_error("LBVH node count mismatch");
      impl_->lbvhTris += B.triCount; impl_->lbvhNodes += wrote;
    }
    CK(cudaEventRecord(impl_->lbvhEv[1], st)); CK(cudaStreamSynchronize(st)); CK(cudaGetLastError()); CK(cudaEventElapsedTime(&impl_->lbvhMs, impl_->lbvhEv[0], impl_->lbvhEv[1]));
    impl_->lbvhNode32Buf.ensure(n0 + extra, st);
    k_nodes32<<<(unsigned)((n0 + extra + 255) / 256), 256, 0, st>>>(ln, (long long)(n0 + extra), impl_->lbvhNode32Buf.p); ++g_kernelLaunches;
    CK(cudaStreamSynchronize(st)); CK(cudaGetLastError());
    d.fnodes = ln; d.fnodes32 = impl_->lbvhNode32Buf.p; d.tris = lt;
  }
  // Kernel variant for this scene shape (dev_isect.cuh TF_*).  Only a speed choice: whatever a lean variant cannot serve is deferred, ray by
  // ray, to the generic kernels, which implement the same rules.
  {
    bool accelInst = false, nonFast = false, nonFastInst = false;
    for (const FBvh& B : hs.bvhs) if (!B.fast) nonFast = true;
    for (const FInstance& in : hs.instances) if (in.baseKind == OK_LIST || in.baseKind == OK_BVH) { accelInst = true; if (in.baseKind == OK_LIST || !hs.bvhs[in.baseIdx].fast) nonFastInst = true; }
    if (d.accelMode == 0 || nonFastInst) impl_->shape = TF_ALL;
    else if (accelInst || nonFast) impl_->shape = TF_LITERAL1;
    else impl_->shape = 0;
    if (const char* f = getenv("DRT_FORCE_SHAPE")) impl_->shape = atoi(f) & TF_ALL;      // tuning / test aid: every shape must give the same image
    impl_->anySecondary = false; for (const FShader& sh : hs.shaders) if (sh.flags & SF_HAS_CAUSTIC) impl_->anySecondary = true;
    if (!keepDepthHint_) { impl_->depthHint = 0; impl_->capHint = 0; }
  }
  impl_->sceneBytes = A.used;                              // bytes copied host -> device by this upload
  d.g = hs.g; d.g.pad0 = 0;
  for (const FPrim& p : hs.prims) if (p.type == PT_MOVSPHERE) d.g.pad0 = 1;
  d.numPhotons = 0; d.phPos = nullptr; d.phPwr = nullptr; d.cellStart = nullptr; d.phPos32 = nullptr; d.phAbsMax = 0; d.padP = 0;
  g_ = d.g;
  impl_->photons.reset();
  CK(cudaStreamSynchronize(st));
}

static inline unsigned gridFor(long long n, int block) { return (unsigned)((n + block - 1) / block); }

// Kernel launches of one call on `st`: counts them into *launches and, with DRT_SYNC_DEBUG set, synchronises after each one (debugging aid:
// locate a faulting kernel).  operator(): one closest-hit or light pass -- the generic kernel alone (lean == null), or the lean kernel, which
// appends what it defers to `list`, followed by the generic kernel as the fix-up pass over that list.  args: the kernels' arguments before
// (work, deferOut).
struct PassLauncher {
  cudaStream_t st; unsigned fixGrid; unsigned long long* launches;
  void launched(const char* what, int level, const char* variant = "") const {
    ++*launches;
    static const bool syncDebug = getenv("DRT_SYNC_DEBUG") != nullptr;
    if (!syncDebug) return;
    cudaError_t e = cudaStreamSynchronize(st); if (e == cudaSuccess) e = cudaGetLastError();
    if (e != cudaSuccess) throw std::runtime_error(std::string("DRT_SYNC_DEBUG: ") + what + variant + " level " + std::to_string(level) + ": " + cudaGetErrorString(e));
  }
  template <class K, class... A> void operator()(const char* what, int level, K lean, K all, uint32_t* list, unsigned grid, A... args) const {
    if (!lean) { all<<<grid, 128, 0, st>>>(args..., nullptr, nullptr); launched(what, level, " generic"); return; }
    lean<<<grid, 128, 0, st>>>(args..., nullptr, list); launched(what, level, " lean");
    all<<<fixGrid, 128, 0, st>>>(args..., list, nullptr); launched(what, level, " fix-up");
  }
};

void Renderer::renderRange(long long pix0, long long pix1, const RenderOutputs& out, RenderStats* stats) { renderChunks(pix0, pix1, 1, 0, 0, out, stats); }

// world > 1: compact pixel p of this rank maps to interleaved row chunks (chunkRows rows each, chunk c of the rank = absolute chunk c*world+rank)
//
// One frame = batches of <= batchRays primary rays; one batch = bounce levels 0..L-1, each {closest hit, surface, [photon gather], lights}, then
// the bottom-up resolve and the pixel pack.  Nothing on this path waits for the device: the length of every level lives in device memory
// (Counters::levelCount), kernels of levels >= 1 run as grid-stride loops over it, and the one host sync of the call is at its end, where the
// device error word says whether the speculation held (queue capacity, launched depth); if not, the frame is rendered again with safer settings.
void Renderer::renderChunks(long long pix0, long long pix1, int world, int rank, int chunkRows, const RenderOutputs& out, RenderStats* stats) {
  CK(cudaSetDevice(device_)); cudaStream_t st = (cudaStream_t)stream_; Impl& I = *impl_;
  PixMap pm; pm.totalPix = (long long)g_.cols * g_.rows; pm.world = world < 1 ? 1 : world; pm.rank = rank; pm.narrow = 0;
  pm.chunkPix = (pm.world == 1) ? (pm.totalPix > 0 ? pm.totalPix : 1) : (long long)chunkRows * g_.cols;
  if (pm.world > 1) { long long nChunks = (g_.rows + chunkRows - 1) / chunkRows, mine = (nChunks - rank + world - 1) / world; pix0 = 0; pix1 = mine * pm.chunkPix; }
  if (!I.ds.prims) throw std::runtime_error("render called before a scene was uploaded");
  const unsigned long long buildLaunches0 = g_kernelLaunches;
  if (g_.photonKind != 0 && !I.photons.built) { devErrorReset(st); if (!I.photons.emitted) I.photons.emitRange(I.ds, 0, g_.numPhotonsCast, I.ctr, I.ctrHost, st); I.photons.buildGrid(I.ds, st); devErrorCheck(st); }
  const int spp = g_.spp < 1 ? 1 : g_.spp;
  const int fullDepth = I.anySecondary ? std::max(1, std::min(g_.numRays - 1, DRT_MAX_LEVELS)) : 1;      // children spawn while gen < numRays - 2
  // kernels of the closest-hit and light passes: the generic kernel alone (counters on, or a scene shape only it serves), or a lean variant
  // followed by the generic kernel as the fix-up pass over what the lean one deferred
  using TraceK = decltype(&k_trace<false, TF_ALL>); using LightK = decltype(&k_light<false, TF_ALL>);
  const TraceK traceAll = counters_ ? &k_trace<true, TF_ALL> : &k_trace<false, TF_ALL>, traceLean = counters_ ? nullptr : I.lean(&k_trace<false, 0>, &k_trace<false, TF_LITERAL1>);
  const LightK lightAll = counters_ ? &k_light<true, TF_ALL> : &k_light<false, TF_ALL>, lightLean = counters_ ? nullptr : I.lean(&k_light<false, 0>, &k_light<false, TF_LITERAL1>);
  long long batchRays = batchRays_; int levels = (I.depthHint > 0) ? std::min(fullDepth, I.depthHint + 1) : fullDepth;
  // queue capacity of a level relative to the batch's primary rays.  2 is the true bound for level 1 and ample for every shipped scene; the true
  // bound of level L is 2^L (binary Fresnel splits), so an overflow doubles the factor (and halves the batch: same memory) and renders again
  double capFactor = std::max(2.0, I.capHint);
  if (const char* e = getenv("DRT_QUEUE_FACTOR")) capFactor = std::max(1e-3, atof(e));      // test aid: force the overflow path
  if (const char* e = getenv("DRT_DEPTH_HINT")) levels = std::max(1, std::min(fullDepth, atoi(e)));    // test aid: force the depth-speculation path
  RenderStats rs; unsigned retries = 0;
  while (true) {
    std::memset(&rs, 0, sizeof(rs)); rs.photonsStored = I.photons.count; rs.photonSeg = I.photons.segments;
    long long pixPerBatch = batchRays / spp; if (pixPerBatch < 1) pixPerBatch = 1;
    const long long maxN0 = std::min(pixPerBatch, std::max<long long>(pix1 - pix0, 1)) * spp;
    // compact pixels are < pix1, so absolute pixels are < (pix1 / chunkPix + 1) * world * chunkPix
    pm.narrow = (maxN0 <= INT32_MAX && (pix1 / pm.chunkPix + 1) * pm.world * pm.chunkPix <= INT32_MAX) ? 1 : 0;
    const long long rayCap = (levels > 1) ? std::max<long long>(64, (long long)(capFactor * (double)maxN0)) : 1;
    const long long nodeCap = (levels > 1) ? maxN0 + ((capFactor >= 64.0) ? 126 * maxN0 : std::max<long long>(64, (long long)(3.0 * capFactor * (double)maxN0))) : maxN0;
    I.hits0.ensure(maxN0, st); I.surf.ensure(std::max(maxN0, rayCap), st); I.nodes.ensure(nodeCap, st);
    if (levels > 1) { I.rays[0].ensure(rayCap, st); I.rays[1].ensure(rayCap, st); I.hits.ensure(rayCap, st); }
    if (traceLean) { I.deferT.ensure(std::max(maxN0, rayCap), st); I.deferL.ensure(std::max(maxN0, rayCap), st); }
    const unsigned persist = (unsigned)std::min<long long>(gridFor(rayCap, 128), (long long)I.numSMs * 16), fixGrid = (unsigned)I.numSMs * 4;
    devErrorReset(st);
    CK(cudaMemsetAsync(I.ctr, 0, sizeof(Counters), st));
    // one closest-hit or light pass of a level; `list` receives what the lean kernel defers
    const PassLauncher pass{st, fixGrid, &rs.kernelLaunches};
    auto launched = [&](const char* what, int level) { pass.launched(what, level); };
    size_t evN = 0; std::vector<size_t> evIdx;      // 4 events per (batch, level): before trace, after trace, after shade (+gather), after light
    CK(cudaEventRecord(I.pev(evN), st)); const size_t evStart = evN++;
    for (long long b0 = pix0; b0 < pix1; b0 += pixPerBatch) {
      const long long nPix = std::min(pixPerBatch, pix1 - b0), n0 = nPix * spp;
      auto wave = [&](int level) { Wave w; w.n0 = n0; w.rayCap = rayCap; w.nodeCap = nodeCap; w.level = level; w.launchedLevels = levels; return w; };
      CK(cudaMemsetAsync(&I.ctr->levelCount, 0, sizeof(Counters) - offsetof(Counters, levelCount), st));
      for (int level = 0; level < levels; ++level) {
        const Wave w = wave(level);
        const RayRec* rays = (level == 0) ? nullptr : I.rays[level & 1].p; RayRec* nextRays = I.rays[(level + 1) & 1].p;
        Hit* hitBuf = (level == 0) ? I.hits0.p : I.hits.p;
        const unsigned grid = (level == 0) ? gridFor(n0, 128) : persist;
        CK(cudaEventRecord(I.pev(evN), st)); evIdx.push_back(evN++);
        pass("k_trace", level, traceLean, traceAll, I.deferT.p, grid, I.ds, w, pm, b0, rays, hitBuf, I.ctr);
        CK(cudaEventRecord(I.pev(evN++), st));
        if (level == 0) k_shade<true><<<grid, 128, 0, st>>>(I.ds, w, pm, b0, rays, hitBuf, I.surf.p, I.nodes.p, nextRays, I.ctr);
        else k_shade<false><<<grid, 128, 0, st>>>(I.ds, w, pm, b0, rays, hitBuf, I.surf.p, I.nodes.p, nextRays, I.ctr);
        launched("k_shade", level);
        if (I.ds.numPhotons > 0) {
          k_photon_gather_lane<<<grid, 128, 0, st>>>(I.ds, w, I.surf.p, I.nodes.p, I.ctr); launched("k_photon_gather_lane", level);
          k_photon_gather_warp<<<grid, 128, 0, st>>>(I.ds, w, I.surf.p, I.nodes.p, I.ctr); launched("k_photon_gather_warp", level);
        }
        CK(cudaEventRecord(I.pev(evN++), st));
        pass("k_light", level, lightLean, lightAll, I.deferL.p, grid, I.ds, w, I.surf.p, I.nodes.p, I.ctr);
        CK(cudaEventRecord(I.pev(evN++), st));
      }
      for (int level = levels - 1; level >= 1; --level) { k_resolve<<<persist, 256, 0, st>>>(wave(level), I.nodes.p, I.ctr); launched("k_resolve", level); }
      k_finish<<<gridFor(nPix, 256), 256, 0, st>>>(I.ds, pm, b0, nPix, I.nodes.p, I.hits0.p, out); launched("k_finish", 0);
    }
    CK(cudaEventRecord(I.pev(evN), st)); const size_t evEnd = evN++;
    CK(cudaMemcpyAsync(I.ctrHost, I.ctr, sizeof(Counters), cudaMemcpyDeviceToHost, st));
    unsigned int devErr = 0; devErrorFetch(&devErr, st);
    CK(cudaStreamSynchronize(st)); CK(cudaGetLastError()); ++rs.hostSyncs;
    throwIfIncomplete(devErr);
    if (devErr & DEV_ERR_DEPTH) { if (levels >= fullDepth) throw std::runtime_error("internal error: bounce depth beyond numRays"); levels = fullDepth; ++retries; continue; }
    if (devErr & DEV_ERR_QUEUE) { if (capFactor >= 64.0) throw std::runtime_error("internal error: secondary-ray queues overflow at their upper bound"); capFactor = std::min(64.0, capFactor * 2); if (capFactor > 2.0) batchRays = std::max<long long>(65536, batchRays / 2); ++retries; continue; }
    float msT = 0, msS = 0, msL = 0, tot = 0;
    for (size_t k : evIdx) { float a, b2, c; CK(cudaEventElapsedTime(&a, I.evPool[k], I.evPool[k + 1])); CK(cudaEventElapsedTime(&b2, I.evPool[k + 1], I.evPool[k + 2])); CK(cudaEventElapsedTime(&c, I.evPool[k + 2], I.evPool[k + 3])); msT += a; msS += b2; msL += c; }
    CK(cudaEventElapsedTime(&tot, I.evPool[evStart], I.evPool[evEnd]));
    const Counters& C = *I.ctrHost;
    for (int k = 0; k < 64; ++k) { rs.primary += C.primaryS[k]; rs.shadow += C.shadowS[k]; }
    rs.primary += C.primary; rs.shadow += C.shadow; rs.reflect += C.reflect; rs.refract += C.refract; rs.boxTests += C.box; rs.primTests += C.prim; rs.boxTestsClosest += C.boxC; rs.primTestsClosest += C.primC;
    rs.deferred = C.deferredTotal; rs.retries = retries;
    I.capHint = capFactor;
    I.depthHint = std::max(1, (int)C.maxLevel + 1);          // levels that held rays this frame: the next frame of this scene launches one more than that
    rs.kernelLaunches += g_kernelLaunches - buildLaunches0;      // photon emission / grid build done inside this call
    rs.msTrace = msT; rs.msShade = msS; rs.msLight = msL; rs.msTotal = tot; rs.msOther = tot - msT - msS - msL;
    break;
  }
  if (stats) *stats = rs;
}

void Renderer::renderToHost(int32_t* argbHost, int32_t* hitPrimHost, int32_t* hitInstHost, double* rgbHost, double* tHost, RenderStats* stats) {
  CK(cudaSetDevice(device_)); cudaStream_t st = (cudaStream_t)stream_; Impl& I = *impl_;
  size_t np = (size_t)g_.cols * g_.rows; RenderOutputs o; std::memset(&o, 0, sizeof(o));
  if (argbHost) { I.oArgb.ensure(np, st); o.argb = I.oArgb.p; } if (hitPrimHost) { I.oPrim.ensure(np, st); o.hitPrim = I.oPrim.p; }
  if (hitInstHost) { I.oInst.ensure(np, st); o.hitInst = I.oInst.p; } if (rgbHost) { I.oRgb.ensure(3 * np, st); o.rgb = I.oRgb.p; } if (tHost) { I.oT.ensure(np, st); o.t = I.oT.p; }
  renderRange(0, (long long)np, o, stats);
  if (argbHost) CK(cudaMemcpyAsync(argbHost, o.argb, np * 4, cudaMemcpyDeviceToHost, st));
  if (hitPrimHost) CK(cudaMemcpyAsync(hitPrimHost, o.hitPrim, np * 4, cudaMemcpyDeviceToHost, st));
  if (hitInstHost) CK(cudaMemcpyAsync(hitInstHost, o.hitInst, np * 4, cudaMemcpyDeviceToHost, st));
  if (rgbHost) CK(cudaMemcpyAsync(rgbHost, o.rgb, np * 24, cudaMemcpyDeviceToHost, st));
  if (tHost) CK(cudaMemcpyAsync(tHost, o.t, np * 8, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
}

double hostPhiloxU01(uint64_t seed, uint32_t stream, uint32_t a, uint32_t b, uint32_t c, uint32_t d) { return philoxU01(seed, stream, a, b, c, d); }
void Renderer::emitPhotons(RenderStats* stats) {
  CK(cudaSetDevice(device_)); Impl& I = *impl_; const unsigned long long l0 = g_kernelLaunches;
  devErrorReset((cudaStream_t)stream_);
  if (g_.photonKind != 0 && !I.photons.built) I.photons.emitAndBuild(I.ds, I.ctr, I.ctrHost, (cudaStream_t)stream_);
  devErrorCheck((cudaStream_t)stream_);
  if (stats) { stats->kernelLaunches = g_kernelLaunches - l0; stats->photonsStored = I.photons.count; stats->photonSeg = I.photons.segments; stats->msTrace = I.photons.msEmit; stats->msOther = I.photons.msBuild; stats->msTotal = I.photons.msEmit + I.photons.msBuild; }
}
// multi-GPU split: emit photon indices [i0, i1) of every light (no grid build); export / import the canonical-order records on the device
void Renderer::emitPhotonsRange(long long i0, long long i1, RenderStats* stats) {
  CK(cudaSetDevice(device_)); Impl& I = *impl_;
  if (g_.photonKind == 0) { I.photons.reset(); return; }
  if (i0 < 0 || i1 > g_.numPhotonsCast || i0 > i1) throw std::runtime_error("photon index range outside [0, photons cast]");
  const unsigned long long l0 = g_kernelLaunches;
  devErrorReset((cudaStream_t)stream_);
  I.photons.emitRange(I.ds, i0, i1, I.ctr, I.ctrHost, (cudaStream_t)stream_);
  devErrorCheck((cudaStream_t)stream_);
  if (stats) { stats->kernelLaunches = g_kernelLaunches - l0; stats->photonsStored = I.photons.count; stats->photonSeg = I.photons.segments; stats->msTrace = I.photons.msEmit; stats->msTotal = I.photons.msEmit; }
}
long long Renderer::exportPhotonsDevice(double* dst6Dev, long long cap) {
  CK(cudaSetDevice(device_)); Impl& I = *impl_; cudaStream_t st = (cudaStream_t)stream_;
  long long n = std::min<long long>((long long)I.photons.count, cap);
  if (n > 0 && dst6Dev) { CK(cudaMemcpyAsync(dst6Dev, I.photons.rec.p, (size_t)n * sizeof(PhotonRec), cudaMemcpyDeviceToDevice, st)); CK(cudaStreamSynchronize(st)); }
  return (long long)I.photons.count;
}
void Renderer::buildPhotonsFromDevice(const double* src6Dev, long long n, RenderStats* stats) {
  CK(cudaSetDevice(device_)); Impl& I = *impl_; cudaStream_t st = (cudaStream_t)stream_;
  if (n < 0 || (n > 0 && !src6Dev)) throw std::runtime_error("bad photon record buffer");
  const unsigned long long l0 = g_kernelLaunches;
  I.photons.setRecords(reinterpret_cast<const PhotonRec*>(src6Dev), (unsigned long long)n, st); I.photons.buildGrid(I.ds, st);
  if (stats) { stats->kernelLaunches = g_kernelLaunches - l0; stats->photonsStored = I.photons.count; stats->msOther = I.photons.msBuild; stats->msTotal = I.photons.msBuild; }
}
// Parity probes: n items, each input and output `w` doubles per item (at most two of each), through the renderer's grow-only probe buffers.
// Resets the device error word, uploads the inputs, zeroes the outputs, runs launch(in, out), downloads the outputs, synchronises once and
// fails the call if a device search ran beyond its capacity.
struct ProbeIn { const void* host; size_t w; };
struct ProbeOut { void* host; size_t w; };
template <class L> static void probe(Renderer::Impl& I, cudaStream_t st, long long n, std::initializer_list<ProbeIn> ins, std::initializer_list<ProbeOut> outs, L launch) {
  double* in[2] = {nullptr, nullptr}; double* out[2] = {nullptr, nullptr}; int k = 0;
  devErrorReset(st);
  for (const ProbeIn& a : ins) { in[k] = I.probeIn[k].ensure(n * a.w, st); CK(cudaMemcpyAsync(in[k], a.host, n * a.w * 8, cudaMemcpyHostToDevice, st)); ++k; }
  k = 0; for (const ProbeOut& a : outs) { out[k] = I.probeOut[k].ensure(n * a.w, st); CK(cudaMemsetAsync(out[k], 0, n * a.w * 8, st)); ++k; }
  launch(in, out);
  k = 0; for (const ProbeOut& a : outs) { CK(cudaMemcpyAsync(a.host, out[k], n * a.w * 8, cudaMemcpyDeviceToHost, st)); ++k; }
  unsigned int e = 0; devErrorFetch(&e, st);
  CK(cudaStreamSynchronize(st)); CK(cudaGetLastError()); throwIfIncomplete(e);
}
void Renderer::probePhotons(long long n, const double* ptsHost, double* out5Host) {
  CK(cudaSetDevice(device_)); Impl& I = *impl_; cudaStream_t st = (cudaStream_t)stream_;
  if (g_.photonKind != 0 && !I.photons.built) { devErrorReset(st); I.photons.emitAndBuild(I.ds, I.ctr, I.ctrHost, st); devErrorCheck(st); }
  probe(I, st, n, {{ptsHost, 3}}, {{out5Host, 5}}, [&](double* const* in, double* const* o) { if (I.ds.numPhotons > 0) k_photon_probe<<<gridFor(n, 128), 128, 0, st>>>(I.ds, n, in[0], o[0]); });
}
// parity probe: the resident packed triangles of fast BVH `fastIndex` and, in DRT_ACCEL_LBVH mode, its GPU-built nodes
long long Renderer::probeFastBvh(int fastIndex, std::vector<FTri>& tris, std::vector<FNode>& nodes, int32_t info[4]) {
  CK(cudaSetDevice(device_)); cudaStream_t st = (cudaStream_t)stream_; int k = 0;
  for (const FBvh& B : impl_->bvhsUploaded) if (B.fast && k++ == fastIndex) {
    tris.resize((size_t)B.triCount); if (B.triCount) CK(cudaMemcpyAsync(tris.data(), impl_->ds.tris + B.triStart, tris.size() * sizeof(FTri), cudaMemcpyDeviceToHost, st));
    const bool lb = impl_->ds.accelMode == 2 && B.fastRoot != B.root; const int nn = lb ? (B.triCount + 3) / 4 - 1 : 0;
    nodes.resize((size_t)nn); if (nn) CK(cudaMemcpyAsync(nodes.data(), impl_->ds.fnodes + B.fastRoot, nodes.size() * sizeof(FNode), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st)); info[0] = B.triStart; info[1] = B.fastRoot; info[2] = nn; info[3] = lb ? 1 : 0; return B.triCount;
  }
  return -1;
}
void Renderer::accelInfo(double out[4]) const { out[0] = impl_->lbvhMs; out[1] = (double)impl_->lbvhTris; out[2] = (double)impl_->lbvhNodes; out[3] = (double)impl_->sceneBytes; }
long long Renderer::getPhotons(double* out6Host, long long cap) { CK(cudaSetDevice(device_)); return impl_->photons.download(out6Host, cap, (cudaStream_t)stream_); }

// parity probe of the closest-hit search: host arrays through the generic query kernel alone (no tmax, hit point or normal, no deferral)
void Renderer::traceRays(long long n, const double* orgHost, const double* dirHost, int32_t* idsHost, double* tHost) {
  CK(cudaSetDevice(device_)); cudaStream_t st = (cudaStream_t)stream_; Impl& I = *impl_;
  probe(I, st, n, {{orgHost, 3}, {dirHost, 3}}, {{idsHost, 1}, {tHost, 1}},       // ids: two int32 per ray
        [&](double* const* in, double* const* o) {
          k_query_closest<TF_ALL><<<gridFor(n, 128), 128, 0, st>>>(I.ds, n, in[0], in[1], nullptr, reinterpret_cast<int32_t*>(o[0]), o[1], nullptr, nullptr, I.ctr, nullptr, nullptr);
        });
}
// Caller rays against the uploaded scene, device arrays in and out.  The rays run through the scene's kernel variant (Impl::shape) with the
// generic kernel as the fix-up pass, in launches of at most 2^31 - 1 rays (the deferral list holds 32-bit indices); one host sync at the end,
// after which the device error word is checked.  Uses the renderer's counters and deferral list as scratch; the frame speculation (depth and
// capacity hints) and the photon map are not touched.  launch(pass, lean, i0, m) queues the pass of rays [i0, i0 + m).
template <class L> static void runQuery(Renderer::Impl& I, cudaStream_t st, long long n, DBuf<uint32_t>& list, bool lean, double RenderStats::*ms, RenderStats* stats, L launch) {
  RenderStats rs; std::memset(&rs, 0, sizeof(rs));
  if (n > 0) {
    const long long per = std::min<long long>(n, INT32_MAX);
    if (lean) list.ensure((size_t)per, st);
    const PassLauncher pass{st, (unsigned)I.numSMs * 4, &rs.kernelLaunches};
    devErrorReset(st);
    CK(cudaMemsetAsync(I.ctr, 0, sizeof(Counters), st));
    CK(cudaEventRecord(I.pev(0), st));
    for (long long i0 = 0; i0 < n; i0 += per) {
      if (i0 > 0) CK(cudaMemsetAsync(&I.ctr->levelCount, 0, sizeof(Counters) - offsetof(Counters, levelCount), st));
      launch(pass, i0, std::min(per, n - i0));
    }
    CK(cudaEventRecord(I.pev(1), st));
    CK(cudaMemcpyAsync(I.ctrHost, I.ctr, sizeof(Counters), cudaMemcpyDeviceToHost, st));
    unsigned int e = 0; devErrorFetch(&e, st);
    CK(cudaStreamSynchronize(st)); CK(cudaGetLastError()); ++rs.hostSyncs;
    throwIfIncomplete(e);
    float t = 0; CK(cudaEventElapsedTime(&t, I.pev(0), I.pev(1)));
    rs.*ms = t; rs.msTotal = t; rs.deferred = I.ctrHost->deferredTotal;
  }
  if (stats) *stats = rs;
}
void Renderer::queryClosest(long long n, const double* org, const double* dir, const double* tmax, int32_t* ids, double* t, double* pos, double* nrm, RenderStats* stats) {
  CK(cudaSetDevice(device_)); Impl& I = *impl_; cudaStream_t st = (cudaStream_t)stream_;
  const auto all = &k_query_closest<TF_ALL>, lean = I.lean(&k_query_closest<0>, &k_query_closest<TF_LITERAL1>);
  runQuery(I, st, n, I.deferT, lean != nullptr, &RenderStats::msTrace, stats, [&](const PassLauncher& pass, long long i0, long long m) {
    pass("k_query_closest", 0, lean, all, I.deferT.p, gridFor(m, 128), I.ds, m, org + 3 * i0, dir + 3 * i0, tmax ? tmax + i0 : nullptr, ids + 2 * i0, t + i0,
         pos ? pos + 3 * i0 : nullptr, nrm ? nrm + 3 * i0 : nullptr, I.ctr);
  });
}
void Renderer::queryOccluded(long long n, const double* org, const double* dir, const double* dist, uint8_t* occluded, RenderStats* stats) {
  CK(cudaSetDevice(device_)); Impl& I = *impl_; cudaStream_t st = (cudaStream_t)stream_;
  const auto all = &k_query_any<TF_ALL>, lean = I.lean(&k_query_any<0>, &k_query_any<TF_LITERAL1>);
  runQuery(I, st, n, I.deferL, lean != nullptr, &RenderStats::msLight, stats, [&](const PassLauncher& pass, long long i0, long long m) {
    pass("k_query_any", 0, lean, all, I.deferL.p, gridFor(m, 128), I.ds, m, org + 3 * i0, dir + 3 * i0, dist + i0, occluded + i0, I.ctr);
  });
}
void Renderer::evalTexture(int shaderIdx, long long n, const double* hitLocHost, const double* fwdLocHost, double* outHost) {
  CK(cudaSetDevice(device_)); cudaStream_t st = (cudaStream_t)stream_;
  probe(*impl_, st, n, {{hitLocHost, 3}, {fwdLocHost, 3}}, {{outHost, 3}},
        [&](double* const* in, double* const* o) { k_eval_texture<<<gridFor(n, 128), 128, 0, st>>>(impl_->ds, shaderIdx, n, in[0], in[1], o[0]); });
}

// ---------------------------------------------------------------------------------------------------------------
// Multi-GPU inside the library (SURVEY 8(b)/(e)): one context per GPU, the frame split in interleaved row chunks, photon emission split by
// photon index.  The only exchanges are an all-gather of photon records and a gather of finished chunks to rank 0, both NCCL calls on the
// renderer's own stream.  NCCL is bound at run time (dlopen): a single-GPU host never needs it.
// ---------------------------------------------------------------------------------------------------------------
}  // namespace drt
#include <dlfcn.h>
#include <nccl.h>
namespace drt {

struct NcclApi {
  void* h = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr; ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr; ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*Send)(const void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr; ncclResult_t (*Recv)(void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*GroupStart)() = nullptr; ncclResult_t (*GroupEnd)() = nullptr; const char* (*GetErrorString)(ncclResult_t) = nullptr;
};
static NcclApi& nccl() {
  static NcclApi a;
  if (!a.h) {
    const char* names[] = {getenv("DRT_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
    for (const char* n : names) { if (!n) continue; a.h = dlopen(n, RTLD_NOW | RTLD_GLOBAL); if (a.h) break; }
    if (!a.h) throw std::runtime_error(std::string("NCCL not found (libnccl.so.2): multi-GPU rendering needs it: ") + dlerror());
    auto sym = [&](const char* n) { void* p = dlsym(a.h, n); if (!p) throw std::runtime_error(std::string("NCCL symbol missing: ") + n); return p; };
    a.GetUniqueId = (decltype(a.GetUniqueId))sym("ncclGetUniqueId"); a.CommInitRank = (decltype(a.CommInitRank))sym("ncclCommInitRank"); a.CommDestroy = (decltype(a.CommDestroy))sym("ncclCommDestroy");
    a.Send = (decltype(a.Send))sym("ncclSend"); a.Recv = (decltype(a.Recv))sym("ncclRecv"); a.AllGather = (decltype(a.AllGather))sym("ncclAllGather");
    a.GroupStart = (decltype(a.GroupStart))sym("ncclGroupStart"); a.GroupEnd = (decltype(a.GroupEnd))sym("ncclGroupEnd"); a.GetErrorString = (decltype(a.GetErrorString))sym("ncclGetErrorString");
  }
  return a;
}
#define NK(x) do { ncclResult_t r_ = (x); if (r_ != ncclSuccess) throw std::runtime_error(std::string("NCCL error: ") + nccl().GetErrorString(r_) + " at " #x); } while (0)

void Renderer::commUniqueId(unsigned char id128[128]) { static_assert(sizeof(ncclUniqueId) == 128, "id size"); ncclUniqueId id; NK(nccl().GetUniqueId(&id)); std::memcpy(id128, &id, 128); }
void Renderer::commInit(const unsigned char id128[128], int world, int rank) {
  if (world < 1 || rank < 0 || rank >= world) throw std::runtime_error("bad world / rank");
  commDestroy(); world_ = world; rank_ = rank;
  if (world == 1) return;
  CK(cudaSetDevice(device_)); ncclUniqueId id; std::memcpy(&id, id128, 128); ncclComm_t c = nullptr;
  NK(nccl().CommInitRank(&c, world, id, rank)); comm_ = c;
}
void Renderer::commDestroy() { if (comm_) { cudaSetDevice(device_); nccl().CommDestroy((ncclComm_t)comm_); comm_ = nullptr; } world_ = 1; rank_ = 0; }

// chunk c of rank r (compact slot j = c * chunkPix + within) -> absolute pixel ((c * world + r) * chunkPix + within)
__global__ void k_unpack_chunks(const int32_t* __restrict__ staging, long long perRankPix, int world, long long chunkPix, long long totalPix, int32_t* __restrict__ frame) {
  const long long n = perRankPix * (world - 1);
  for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (long long)gridDim.x * blockDim.x) {
    const int r = 1 + (int)(k / perRankPix); const long long j = k % perRankPix, c = j / chunkPix, within = j % chunkPix;
    const long long q = (c * world + r) * chunkPix + within;
    if (q < totalPix) frame[q] = staging[(long long)(r - 1) * perRankPix + j];
  }
}
__global__ void k_store_u64(unsigned long long* dst, unsigned long long v) { *dst = v; }

long long Renderer::distRankPixels(int cols, int rows, int world, int rank, int chunkRows) {
  const long long nChunks = (rows + chunkRows - 1) / chunkRows; return ((nChunks - rank + world - 1) / world) * (long long)chunkRows * cols;
}
long long Renderer::distAbsPixel(int cols, int rows, int world, int rank, int chunkRows, long long compact) {
  PixMap pm; pm.totalPix = (long long)cols * rows; pm.world = world; pm.rank = rank; pm.narrow = 0; pm.chunkPix = (world == 1) ? std::max<long long>(pm.totalPix, 1) : (long long)chunkRows * cols;
  const long long q = absPixel(pm, compact); return q < pm.totalPix ? q : -1;
}
void Renderer::distPhotonRange(long long nCast, int world, int rank, long long out2[2]) { out2[0] = nCast * rank / world; out2[1] = nCast * (rank + 1) / world; }

void Renderer::renderDistributed(int32_t* argbHostRank0, int32_t* argbDevRank0, int chunkRows, bool reemitPhotons, RenderStats* stats) {
  CK(cudaSetDevice(device_)); cudaStream_t st = (cudaStream_t)stream_; Impl& I = *impl_;
  const int world = world_, rank = rank_; if (chunkRows < 1) chunkRows = 8;
  if (world > 1 && !comm_) throw std::runtime_error("drt_comm_init has not been called on this context");
  const long long totalPix = (long long)g_.cols * g_.rows, chunkPix = (long long)chunkRows * g_.cols;
  const long long nChunks = (g_.rows + chunkRows - 1) / chunkRows, perRankChunks = (nChunks + world - 1) / world, perRankPix = perRankChunks * chunkPix;
  auto chunksOf = [&](int r) { return distRankPixels(g_.cols, g_.rows, world, r, chunkRows) / chunkPix; };
  unsigned long long photonLaunches = 0; float msPhoton = 0;
  // ---- photon pass: rank r emits photon indices [r N / world, (r+1) N / world) of every light; canonical-order records are all-gathered
  //      (counts first, blocks padded to the longest) and every rank builds the full grid: bit-identical to the single-GPU map
  if (g_.photonKind != 0 && (reemitPhotons || !I.photons.built)) {
    const unsigned long long l0 = g_kernelLaunches; cudaEvent_t e0 = I.pev(0), e1 = I.pev(1); CK(cudaEventRecord(e0, st));
    long long pr[2]; distPhotonRange(g_.numPhotonsCast, world, rank, pr); const long long i0 = pr[0], i1 = pr[1];
    devErrorReset(st); I.photons.emitRange(I.ds, i0, i1, I.ctr, I.ctrHost, st); devErrorCheck(st);
    if (world > 1) {
      unsigned long long* cnt = I.xCnt.ensure((size_t)world + 1, st);
      k_store_u64<<<1, 1, 0, st>>>(cnt + world, I.photons.count);
      NK(nccl().AllGather(cnt + world, cnt, 1, ncclUint64, (ncclComm_t)comm_, st));
      std::vector<unsigned long long> counts(world); CK(cudaMemcpyAsync(counts.data(), cnt, sizeof(unsigned long long) * world, cudaMemcpyDeviceToHost, st)); CK(cudaStreamSynchronize(st));
      unsigned long long mx = 1, total = 0, segs = I.photons.segments; for (auto c : counts) { mx = std::max(mx, c); total += c; }
      PhotonRec* mine = I.xMine.ensure((size_t)mx, st); PhotonRec* all = I.xAll.ensure((size_t)mx * world, st);
      CK(cudaMemsetAsync(mine, 0, mx * sizeof(PhotonRec), st));
      if (I.photons.count) CK(cudaMemcpyAsync(mine, I.photons.rec.p, I.photons.count * sizeof(PhotonRec), cudaMemcpyDeviceToDevice, st));
      NK(nccl().AllGather(mine, all, mx * sizeof(PhotonRec), ncclChar, (ncclComm_t)comm_, st));
      I.photons.built = false; I.photons.emitted = true; I.photons.count = 0; I.photons.rec.ensure((size_t)total, st);
      unsigned long long at = 0; for (int r = 0; r < world; ++r) { if (counts[r]) CK(cudaMemcpyAsync(I.photons.rec.p + at, all + (size_t)r * mx, counts[r] * sizeof(PhotonRec), cudaMemcpyDeviceToDevice, st)); at += counts[r]; }
      I.photons.count = total; I.photons.segments = segs; CK(cudaStreamSynchronize(st));
    }
    I.photons.buildGrid(I.ds, st);
    CK(cudaEventRecord(e1, st)); CK(cudaStreamSynchronize(st)); CK(cudaEventElapsedTime(&msPhoton, e0, e1)); photonLaunches = g_kernelLaunches - l0;
  }
  // ---- this rank's chunks: rank 0 renders in place into the frame, the others into a compact buffer that is sent as one message
  RenderOutputs o; std::memset(&o, 0, sizeof(o)); RenderStats rs; std::memset(&rs, 0, sizeof(rs));
  if (rank == 0) { if (argbDevRank0) o.argb = argbDevRank0; else { I.oArgb.ensure((size_t)(perRankPix * world), st); o.argb = I.oArgb.p; } }
  else { I.oArgb.ensure((size_t)perRankPix, st); o.argb = I.oArgb.p; o.packed = 1; }
  if (world == 1) renderChunks(0, totalPix, 1, 0, 0, o, &rs); else renderChunks(0, 0, world, rank, chunkRows, o, &rs);
  if (world > 1) {
    if (rank == 0) {
      I.oPrim.ensure((size_t)(perRankPix * (world - 1)), st);        // staging for the other ranks' compact buffers
      NK(nccl().GroupStart());
      for (int r = 1; r < world; ++r) NK(nccl().Recv(I.oPrim.p + (size_t)(r - 1) * perRankPix, (size_t)(chunksOf(r) * chunkPix), ncclInt32, r, (ncclComm_t)comm_, st));
      NK(nccl().GroupEnd());
      k_unpack_chunks<<<(unsigned)std::min<long long>((perRankPix * (world - 1) + 255) / 256, 148 * 16), 256, 0, st>>>(I.oPrim.p, perRankPix, world, chunkPix, totalPix, o.argb); ++rs.kernelLaunches;
    } else NK(nccl().Send(o.argb, (size_t)(chunksOf(rank) * chunkPix), ncclInt32, 0, (ncclComm_t)comm_, st));
  }
  if (rank == 0 && argbHostRank0) CK(cudaMemcpyAsync(argbHostRank0, o.argb, (size_t)totalPix * 4, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st)); CK(cudaGetLastError());
  rs.kernelLaunches += photonLaunches; rs.msOther += msPhoton; rs.msTotal += msPhoton;
  if (stats) *stats = rs;
}

}  // namespace drt
