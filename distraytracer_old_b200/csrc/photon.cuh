// Photon map on the device: emission + random-walk kernel, uniform-grid build (cell count -> scan -> stable radix sort),
// warp-cooperative k-nearest radiance gather.
//
// Replaces (reference file:line, /root/reference/src/rayTracerDistAccelShdPhtnMap/):
//   k_photon_emit     myScene.java:952-998 sendCausticPhotons, :1000-1091 sendDiffusePhotons (one thread = one emitted photon,
//                     the whole walk of <= numPhotonRays+1 segments in-thread); myLight.java:59-74 getRandDir, :104-107 / :165-185 /
//                     :229-242 genRndPhtnRay; myObjShader.java:461-478 findCausticRayHit, :297-406 calcTransRay / calcReflRay
//   grid build        myLight.java:325-381 myKD_Tree.build_tree (balanced kd-tree) -> uniform grid of cell size >= search radius;
//                     photons sorted by cell with the stable radix sort of dev_sort.cuh, cellStart = exclusive scan of per-cell counts
//   k_photon_gather   myLight.java:389-445 find_near (k nearest with d^2 < r^2, shrinking radius) + myObjShader.java:441-458
//                     getIrradianceFromPhtnTree: sum(power) / (PI_float * d^2 of the farthest of the k).  The set "k nearest inside the
//                     radius" does not depend on the search structure, so the grid returns what the kd-tree returns (exact-distance
//                     ties at the k-th neighbour excepted).
// Photon order is canonical: record order = (photon index, light index, store index), independent of launch geometry and of how
// photon indices are split across GPUs; the per-cell order after the stable sort inherits it, so sums are reproducible.
#pragma once
#include "dbuf.h"
#include "dev_sort.cuh"
#include <algorithm>
#include <vector>

namespace drt {

struct alignas(16) PhotonRec { double x, y, z, r, g, b; };     // 48 B: position (world) + power

// ---------------------------------------------------------------------------------------------------------------
// emission
// ---------------------------------------------------------------------------------------------------------------
struct PhSampler {
  uint64_t seed; uint32_t photon, light;
  __device__ __forceinline__ double u(uint32_t seg, uint32_t dim) const { return philoxU01(seed, STREAM_PHOTON, photon, light, seg, dim); }
};

// Light::getRandDir: rejection-sampled uniform direction (myLight.java:59-74)
__device__ inline D3 phRandDir(const PhSampler& sp, uint32_t& draw) {
  double x, y, z, sq;
  do {
    x = urange(sp.u(0, draw), -1.0, 1.0); y = urange(sp.u(0, draw + 1), -1.0, 1.0); z = urange(sp.u(0, draw + 2), -1.0, 1.0); draw += 3;
    sq = (x * x) + (y * y) + (z * z);
  } while ((sq > 1.0) || (sq < DRT_EPS));
  double mag = sqrt(sq); return d3(x / mag, y / mag, z / mag);
}
__device__ __forceinline__ double phAngleProb(double angle, double inner, double outer, double diff) { return (angle < inner) ? 1 : (angle > outer) ? 0 : (outer - angle) / diff; }

__device__ inline void phGenRay(const DScene& S, const FLight& L, const PhSampler& sp, D3& org, D3& dir) {
  uint32_t draw = 0; const FXform& LX = S.xforms[L.xform];
  D3 lo = d3(L.origin[0], L.origin[1], L.origin[2]), orient = d3(L.orient[0], L.orient[1], L.orient[2]), tang = d3(L.tangent[0], L.tangent[1], L.tangent[2]);
  if (L.type == LT_POINT) { dir = phRandDir(sp, draw); org = xfPoint(LX.m, lo); }
  else if (L.type == LT_SPOT) {
    double prob, angle, checkProb = urange(sp.u(0, draw++), 0, 1);
    do { angle = urange(sp.u(0, draw++), 0, L.outerRad); prob = phAngleProb(angle, L.innerRad, L.outerRad, L.radDiff); } while (prob > checkProb);
    D3 tmp = norm3(rotAboutAxis(orient, tang, angle));
    dir = rotAboutAxis(tmp, orient, urange(sp.u(0, draw++), 0, DRT_TWO_PI_F)); org = xfPoint(LX.m, lo);
  } else {
    double prob, angle;
    do { angle = urange(sp.u(0, draw), 0, DRT_PI); prob = phAngleProb(angle, 0, DRT_PI, DRT_PI); double chk = urange(sp.u(0, draw + 1), 0, 1); draw += 2; if (!(prob > chk)) break; } while (true);
    D3 d = norm3(rotAboutAxis(orient, tang, angle));
    d = rotAboutAxis(d, orient, urange(sp.u(0, draw), 0, DRT_TWO_PI_F));
    double ua = sp.u(0, draw + 1), ur = sp.u(0, draw + 2); draw += 3;
    D3 tmp = norm3(rotAboutAxis(tang, orient, urange(ua, 0, DRT_TWO_PI_F)));
    dir = d; org = xfPoint(LX.m, add3(scale3(tmp, urange(ur, 0, L.radius)), lo));
  }
}

struct PhHit { bool isHit; int shader; int gen; uint32_t seg; double kt0; D3 fwd, nrm, rawDir; };
__device__ __noinline__ void phTrace(const DScene& S, D3 o, D3 dirUnnormalized, int gen, uint32_t seg, double kt0, const PhSampler& sp, PhHit& ph) {
  Ray ray = makeRay(o, norm3(dirUnnormalized)); Hit h;
  double time = S.g.pad0 ? sp.u(seg, 0xFFFFu) : 0.0;
  ph.isHit = closestHit(S, ray, time, h, nullptr); ph.gen = gen; ph.seg = seg; ph.kt0 = kt0; ph.shader = -1;
  if (!ph.isHit) return;
  const FPrim P = S.prims[h.prim]; const FXform& X = S.xforms[h.hitXform];
  ph.shader = h.shaderOverride >= 0 ? h.shaderOverride : P.shader;
  ph.fwd = xfPoint(X.m, h.loc); ph.nrm = norm3(xfVector(X.adj, primNormal(S, P, h.loc, h.arg0, h.arg1, h.state))); ph.rawDir = h.rawDir;
}
// myObjShader.findCausticRayHit: next segment off a specular surface; scales pwr. Returns false when the walk ends here.
__device__ inline bool phSpecular(const DScene& S, const FShader& sh, const PhHit& h, double pwr[3], D3& dir, double& kt0) {
  if (!((h.gen < S.g.numPhotonRays) && (sh.flags & SF_HAS_CAUSTIC))) return false;
  double pm[3] = {1.0, 1.0, 1.0}; bool have = false; kt0 = 1;
  if ((sh.KTrans > 0.0) || (sh.currPerm > 0.0)) {
    pm[0] = sh.phtnPermClr[0]; pm[1] = sh.phtnPermClr[1]; pm[2] = sh.phtnPermClr[2];
    Fres f = fresnel(h.rawDir, h.nrm, sh.KTrans, h.kt0);
    if (f.oneM > DRT_EPS) dir = refractDir(f); else dir = scale3(reflDir(f.back, f.N), f.mult);
    kt0 = sh.KTrans; have = true;
  } else if (sh.KRefl > 0.0) {
    pm[0] = pm[1] = pm[2] = sh.KRefl; dir = reflDir(scale3(h.rawDir, -1), h.nrm); have = true;
  }
  for (int i = 0; i < 3; ++i) pwr[i] = pwr[i] * pm[i];
  return have;
}

// one thread = photon index (i0 + g / numLights) of light (g % numLights); stores go to fixed slots g*maxStore.. and are compacted afterwards
#ifndef DRT_EMIT_MINBLOCKS
#define DRT_EMIT_MINBLOCKS 4      // 128 registers: 16 M photons in 14.7 ms vs 22.9 ms at 255 registers (profiles/r1_tuning.md)
#endif
__global__ void __launch_bounds__(128, DRT_EMIT_MINBLOCKS) k_photon_emit(const __grid_constant__ DScene S, long long i0, long long nThreads, int maxStore, PhotonRec* __restrict__ slots, uint32_t* __restrict__ slotCount, Counters* ctr) {
  long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; unsigned long long segs = 0;
  if (g < nThreads) {
    const int nl = S.g.numLights; PhSampler sp; sp.seed = S.g.seed; sp.photon = (uint32_t)(i0 + g / nl); sp.light = (uint32_t)(g % nl);
    const FLight L = S.lights[sp.light]; const bool caustic = S.g.photonKind == 1;
    const double pwrMult = (caustic ? S.g.causticPwrMult : S.g.diffusePwrMult) / S.g.numPhotonsCast;
    double pwr[3] = {L.color[0] * pwrMult, L.color[1] * pwrMult, L.color[2] * pwrMult};
    PhotonRec* out = slots + g * maxStore; int nStore = 0;
    auto store = [&](const PhHit& h) { if (nStore < maxStore) { PhotonRec r; r.x = h.fwd.x; r.y = h.fwd.y; r.z = h.fwd.z; r.r = pwr[0]; r.g = pwr[1]; r.b = pwr[2]; out[nStore] = r; } ++nStore; };
    D3 o, d; phGenRay(S, L, sp, o, d);
    PhHit h; ++segs; phTrace(S, o, d, 0, 0, 1.0, sp, h);
    if (caustic) {
      if (h.isHit && (S.shaders[h.shader].flags & SF_HAS_CAUSTIC)) {
        int lastGen = 0; bool have;
        do {
          const FShader sh = S.shaders[h.shader]; D3 nd; double kt0;
          have = phSpecular(S, sh, h, pwr, nd, kt0);
          if (have) { lastGen = h.gen + 1; ++segs; phTrace(S, h.fwd, nd, h.gen + 1, h.seg + 1, kt0, sp, h); }
          else h.isHit = false;
        } while (h.isHit && (S.shaders[h.shader].flags & SF_HAS_CAUSTIC) && (lastGen <= S.g.numPhotonRays));
        if (h.isHit && !(lastGen > S.g.numPhotonRays)) store(h);
      }
    } else if (h.isHit) {
      bool done = false, firstDiff = true;
      do {
        const FShader sh = S.shaders[h.shader];
        if (sh.KRefl == 0) {
          double prob = 0; const uint32_t seg = h.seg + 1; uint32_t dr = 0;
          if (!firstDiff) { store(h); prob = urange(sp.u(seg, dr++), 0, 1.0); }
          firstDiff = false;
          if (prob < sh.avgDiff) {
            double x, y, z, sq;
            do { x = urange(sp.u(seg, dr), -1.0, 1.0); y = urange(sp.u(seg, dr + 1), -1.0, 1.0); dr += 2; sq = (x * x) + (y * y); } while ((sq >= 1.0) || (sq < DRT_EPS));
            z = sqrt(1 - (sq));
            D3 n = h.nrm; double nxSq = n.x * n.x, nySq = n.y * n.y, nzSq = n.z * n.z;
            D3 tmpV = ((nxSq > nySq) && (nxSq > nzSq)) ? d3(0, 0, 1) : d3(1, 0, 0);
            D3 p_ = cross3(n, tmpV), q_ = cross3(p_, n);
            n = scale3(n, z); p_ = scale3(p_, x); q_ = scale3(q_, y);
            D3 bd = d3(n.x + p_.x + q_.x, n.y + p_.y + q_.y, n.z + p_.z + q_.z);
            pwr[0] = pwr[0] * sh.phtnDiffScl[0]; pwr[1] = pwr[1] * sh.phtnDiffScl[1]; pwr[2] = pwr[2] * sh.phtnDiffScl[2];
            ++segs; phTrace(S, h.fwd, bd, h.gen + 1, seg, 1.0, sp, h);
          } else done = true;
        } else {
          D3 nd; double kt0;
          if (phSpecular(S, sh, h, pwr, nd, kt0)) { ++segs; phTrace(S, h.fwd, nd, h.gen + 1, h.seg + 1, kt0, sp, h); }
          else h.isHit = false;
        }
      } while (h.isHit && !done && (h.gen <= S.g.numPhotonRays));
    }
    slotCount[g] = (uint32_t)(nStore < maxStore ? nStore : maxStore);
  }
  warpAdd(&ctr->pad, segs);
}

// compaction of the fixed slots into the canonical record order
__global__ void k_photon_compact(long long nThreads, int maxStore, const PhotonRec* __restrict__ slots, const uint32_t* __restrict__ slotCount, const uint32_t* __restrict__ slotOffset, PhotonRec* __restrict__ out) {
  long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; if (g >= nThreads) return;
  uint32_t c = slotCount[g], o = slotOffset[g];
  for (uint32_t i = 0; i < c; ++i) out[o + i] = slots[g * maxStore + i];
}

// ---------------------------------------------------------------------------------------------------------------
// grid build
// ---------------------------------------------------------------------------------------------------------------
struct PhGrid { double gmin[3]; double cell; uint32_t dim[3]; uint32_t nCells; };

__global__ void k_photon_bounds(const PhotonRec* __restrict__ rec, long long n, double* __restrict__ blockMinMax /*[grid][6]*/) {
  double mn[3] = {DRT_DMAX, DRT_DMAX, DRT_DMAX}, mx[3] = {-DRT_DMAX, -DRT_DMAX, -DRT_DMAX};
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const PhotonRec r = rec[i]; double p[3] = {r.x, r.y, r.z};
    for (int k = 0; k < 3; ++k) { mn[k] = fmin(mn[k], p[k]); mx[k] = fmax(mx[k], p[k]); }
  }
  __shared__ double sm[8][6];
  for (int k = 0; k < 3; ++k) for (int o = 16; o > 0; o >>= 1) { mn[k] = fmin(mn[k], __shfl_down_sync(0xffffffffu, mn[k], o)); mx[k] = fmax(mx[k], __shfl_down_sync(0xffffffffu, mx[k], o)); }
  if ((threadIdx.x & 31) == 0) for (int k = 0; k < 3; ++k) { sm[threadIdx.x >> 5][k] = mn[k]; sm[threadIdx.x >> 5][3 + k] = mx[k]; }
  __syncthreads();
  if (threadIdx.x < 3) { double a = sm[0][threadIdx.x], b = sm[0][3 + threadIdx.x]; for (int w = 1; w < (int)(blockDim.x >> 5); ++w) { a = fmin(a, sm[w][threadIdx.x]); b = fmax(b, sm[w][3 + threadIdx.x]); }
    blockMinMax[blockIdx.x * 6 + threadIdx.x] = a; blockMinMax[blockIdx.x * 6 + 3 + threadIdx.x] = b; }
}
__device__ __forceinline__ int phCellCoord(double v, double gmin, double cell, int dim) { int c = (int)floor((v - gmin) / cell); return c < 0 ? 0 : (c >= dim ? dim - 1 : c); }
// Two-level key of fine cell (fx, fy, fz) in a grid of dx x dy x . coarse cells: the coarse cell (side = search radius, x fastest) shifted left
// by 6, OR the 4x4x4 fine sub-cell.  Consecutive keys therefore cover a row of coarse cells along x and a run of fine cells along x inside one
// coarse cell (phRowRange): each is one contiguous photon range of cellStart.
__device__ __forceinline__ uint32_t phKey(uint32_t dx, uint32_t dy, uint32_t fx, uint32_t fy, uint32_t fz) {
  return ((((fz >> 2) * dy + (fy >> 2)) * dx + (fx >> 2)) << 6) | ((fz & 3u) << 4) | ((fy & 3u) << 2) | (fx & 3u);
}
__global__ void k_photon_cellkeys(const PhotonRec* __restrict__ rec, long long n, PhGrid G, uint32_t* __restrict__ keys, uint32_t* __restrict__ cellCount) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; if (i >= n) return;
  const PhotonRec r = rec[i];
  // every coordinate derives from the FINE one, so both levels of the key are consistent with each other
  const double cf = G.cell * 0.25;
  const uint32_t fx = phCellCoord(r.x, G.gmin[0], cf, 4 * G.dim[0]), fy = phCellCoord(r.y, G.gmin[1], cf, 4 * G.dim[1]), fz = phCellCoord(r.z, G.gmin[2], cf, 4 * G.dim[2]);
  const uint32_t key = phKey(G.dim[0], G.dim[1], fx, fy, fz);
  keys[i] = key; atomicAdd(&cellCount[key], 1u);
}
// sorted order -> the two 32-byte-per-photon arrays the gather reads with 128-bit loads
// (+ a float4 mirror of the positions for the gather's FP32 pre-test, see phWarpGather32)
__global__ void k_photon_reorder(const PhotonRec* __restrict__ rec, const uint32_t* __restrict__ order, long long n, double4* __restrict__ pos, double4* __restrict__ pwr, float4* __restrict__ pos32) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; if (i >= n) return;
  const PhotonRec r = rec[order[i]]; pos[i] = make_double4(r.x, r.y, r.z, 0.0); pwr[i] = make_double4(r.r, r.g, r.b, 0.0); pos32[i] = make_float4((float)r.x, (float)r.y, (float)r.z, 0.0f);
}

// ---------------------------------------------------------------------------------------------------------------
// gather
// ---------------------------------------------------------------------------------------------------------------
#define DRT_PH_LANE_MAX 1024u     // candidate count up to which a lane serves its own query
#define DRT_PH_BINS 256
#define DRT_PH_LIST 128
// Candidate ranges of one warp query.  Coarse rows: the cell is >= r, so the bounding cube of a sphere of radius r (1 + 1e-7) touches at most
// 4 cells per axis: <= 4 x 4 rows.  Fine runs: a plan's block is at most 7 fine cells per axis (s <= 3), and 7 consecutive fine cells touch at
// most 3 coarse cells along x: <= 3 x 7 x 7 = 147 runs.
#define DRT_PH_MAXRANGES 160
struct PhWarpShared { uint32_t hist[DRT_PH_BINS]; double listD2[DRT_PH_LIST]; uint32_t listIdx[DRT_PH_LIST]; uint32_t listN; uint32_t pad[3];
                      uint32_t rA[DRT_PH_MAXRANGES + 33], rOff[DRT_PH_MAXRANGES + 33]; };     // non-empty candidate ranges: first photon, exclusive prefix of the lengths (+ sentinels)

// photon range [a, b) of the cells x0..x1 of one row: the coarse cells of coarse row (y, z), or (fine) the fine cells of fine row (y, z), which
// must lie inside one coarse cell (x1 <= x0 | 3)
__device__ __forceinline__ void phRowRange(const DScene& S, bool fine, int y, int z, int x0, int x1, uint32_t& a, uint32_t& b) {
  const uint32_t c = fine ? 1u : 4u;                                        // fine cells per cell of the row
  a = S.cellStart[phKey(S.gridDim[0], S.gridDim[1], c * x0, c * y, c * z)];
  b = S.cellStart[phKey(S.gridDim[0], S.gridDim[1], c * x1, c * y, c * z) + (fine ? 1u : 64u)];     // the key after cell x1
}

// cells the bounding cube of the search sphere overlaps (radius inflated by 1e-7 so that no photon with d^2 < r^2 can sit in a cell outside
// the range whatever the rounding of its own cell index); false when the cube misses the grid
__device__ __forceinline__ bool phCellRange(const DScene& S, D3 p, double radius2, int lo[3], int hi[3]) {
  const double rr = sqrt(radius2) * 1.0000001, cell = S.cellSize; const double pp[3] = {p.x, p.y, p.z}; bool ok = true;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const double a = floor((pp[k] - rr - S.gridMin[k]) / cell), b = floor((pp[k] + rr - S.gridMin[k]) / cell); const int dim = (int)S.gridDim[k];
    if (!(b >= 0) || !(a <= dim - 1)) ok = false;
    lo[k] = a < 0 ? 0 : (a > dim - 1 ? dim - 1 : (int)a); hi[k] = b > dim - 1 ? dim - 1 : (b < 0 ? 0 : (int)b);
  }
  return ok;
}

// ---- warp-cooperative tier: the k nearest photons with d^2 < r^2 around p, their summed power and the largest of their d^2, computed by one
// warp.  The candidates of a query are a list of photon ranges (phWarpRanges); two selections read it, and both end in the same exact
// resolution of a short boundary list by (double d^2, index) (phRankList).

// The candidate ranges -- coarse rows lo..hi, or the runs of fine cells lo..hi (fine) -- enumerated lane-parallel and compacted (empty ones
// dropped) into shared memory with the running offset of each.  Range order = z, then y, then x, so photon order within the list is fixed.
struct PhRanges { uint32_t n, total; };
__device__ inline PhRanges phWarpRanges(const DScene& S, bool fine, const int lo[3], const int hi[3], PhWarpShared& sh) {
  const unsigned lane = threadIdx.x & 31;
  const int x0 = lo[0], x1 = hi[0], y0 = lo[1], z0 = lo[2], nx = fine ? (x1 >> 2) - (x0 >> 2) + 1 : 1, ny = hi[1] - y0 + 1, nz = hi[2] - z0 + 1;
  int slots = nx * ny * nz;
  if (slots > DRT_PH_MAXRANGES) { flagError(DEV_ERR_INCOMPLETE); slots = 0; }      // excluded by the bound above; the host reports an incomplete result
  uint32_t nRanges = 0, total = 0;
  for (int s0 = 0; s0 < slots; s0 += 32) {
    const int slot = s0 + (int)lane; uint32_t a = 0, b = 0;
    if (slot < slots) {
      const int ir = slot % nx, fy = y0 + (slot / nx) % ny, fz = z0 + slot / (nx * ny);
      const int fx = ir == 0 ? x0 : (((x0 >> 2) + ir) << 2);
      phRowRange(S, fine, fy, fz, fx, fine ? min(x1, fx | 3) : x1, a, b);
    }
    const uint32_t len = b - a; const unsigned ne = __ballot_sync(0xffffffffu, len > 0);
    uint32_t incl = len;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= (unsigned)o) incl += t; }
    if (len > 0) { const uint32_t at = nRanges + __popc(ne & ((1u << lane) - 1u)); sh.rA[at] = a; sh.rOff[at] = total + incl - len; }
    nRanges += __popc(ne); total += __shfl_sync(0xffffffffu, incl, 31);
  }
  for (uint32_t i = nRanges + lane; i < nRanges + 33; i += 32) { sh.rA[i] = 0; sh.rOff[i] = total; }       // sentinels: empty ranges at the end
  __syncwarp();
  return {nRanges, total};
}
// f(j, valid) warp-wide for every candidate: range by range, 32 consecutive photons of a range per step
template <class F> __device__ __forceinline__ void phEachRange(const PhWarpShared& sh, PhRanges R, F&& f) {
  const unsigned lane = threadIdx.x & 31;
  for (uint32_t r = 0; r < R.n; ++r) {
    const uint32_t a = sh.rA[r], b = a + (sh.rOff[r + 1] - sh.rOff[r]);
    for (uint32_t j0 = a; j0 < b; j0 += 32) f(j0 + lane, j0 + lane < b);
  }
}
// f(j, valid) warp-wide for every candidate, 32 consecutive FLAT indices per step: a fine row run holds ~10-30 photons, so the per-range walk
// leaves two thirds of the lanes idle and spends 40 % of the instructions on warp-uniform range bookkeeping (profiles/r2d_ncu_gather.md).
// base = range holding flat index t0; the ranges that start inside (t0, t0 + 32) are among the next 32 (every range is non-empty), each lane
// looks at one of them: OR of their start bits -> owner of every lane.
template <class F> __device__ __forceinline__ void phEachFlat(const PhWarpShared& sh, PhRanges R, F&& f) {
  if (R.total >= 64u * R.n) { phEachRange(sh, R, f); return; }      // long ranges (coarse rows of a sparse map): the per-range walk wastes nothing
  const unsigned lane = threadIdx.x & 31; uint32_t base = 0;
  for (uint32_t t0 = 0; t0 < R.total; t0 += 32) {
    const uint32_t rel = sh.rOff[base + 1 + lane] - t0;                      // >= 1
    const unsigned mask = __reduce_or_sync(0xffffffffu, rel < 32u ? (1u << rel) : 0u);
    const uint32_t owner = base + __popc(mask & ((2u << lane) - 1u)), t = t0 + lane;
    f(sh.rA[owner] + (t - sh.rOff[owner]), t < R.total);
    base += __popc(__ballot_sync(0xffffffffu, rel <= 32u));
  }
}
// the histogram bin where the running count reaches `target` (1 <= target <= the histogram's total): its index, the count of the bins below it
// and its own count
__device__ __forceinline__ void phFindBin(const PhWarpShared& sh, uint32_t target, uint32_t& bin, uint32_t& before, uint32_t& inBin) {
  const unsigned lane = threadIdx.x & 31;
  uint32_t loc[8], s = 0;
#pragma unroll
  for (int i = 0; i < 8; ++i) { loc[i] = sh.hist[lane * 8 + i]; s += loc[i]; }
  uint32_t incl = s;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= (unsigned)o) incl += t; }
  const unsigned reach = __ballot_sync(0xffffffffu, incl >= target); const int L = __ffs(reach) - 1;
  bin = 0; before = 0; inBin = 0;
  if ((int)lane == L) { uint32_t c = incl - s; for (int i = 0; i < 8; ++i) { if (c + loc[i] >= target) { bin = lane * 8 + i; before = c; inBin = loc[i]; break; } c += loc[i]; } }
  bin = __shfl_sync(0xffffffffu, bin, L); before = __shfl_sync(0xffffffffu, before, L); inBin = __shfl_sync(0xffffffffu, inBin, L);
}
// exact end of both selections: the `need` smallest (d^2, index) of the boundary list sh.listD2 / listIdx go into the lane's sums
__device__ __forceinline__ void phRankList(const PhWarpShared& sh, int need, const double4* __restrict__ W, double& s0, double& s1, double& s2, double& mx) {
  __syncwarp();
  const int n = (int)min(sh.listN, (uint32_t)DRT_PH_LIST);
  for (int i = threadIdx.x & 31; i < n; i += 32) {
    const double di = sh.listD2[i]; const uint32_t ji = sh.listIdx[i]; int rank = 0;
    for (int t = 0; t < n; ++t) { const double dt = sh.listD2[t]; rank += (dt < di || (dt == di && sh.listIdx[t] < ji)) ? 1 : 0; }
    if (rank < need) { const double4 w = W[ji]; s0 += w.x; s1 += w.y; s2 += w.z; mx = fmax(mx, di); }
  }
}
__device__ __forceinline__ void phWarpSum(double s0, double s1, double s2, double mx, double sum[3], double& dmax2) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) { s0 += __shfl_xor_sync(0xffffffffu, s0, o); s1 += __shfl_xor_sync(0xffffffffu, s1, o); s2 += __shfl_xor_sync(0xffffffffu, s2, o); mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o)); }
  sum[0] = s0; sum[1] = s1; sum[2] = s2; dmax2 = mx;
}

// FP64 selection: radix select on a 32-bit quantisation of d^2 (monotone in d^2), 8 bits per level, each level one walk over the candidates,
// finished exactly on the boundary bin once it holds <= DRT_PH_LIST photons.  r2: search threshold (the scene's r^2, or a smaller guess --
// then `needAll`: return false without a result if fewer than k photons are inside it).
__device__ inline bool phWarpGather64(const DScene& S, D3 p, double r2, bool needAll, PhRanges R, PhWarpShared& sh, double sum[3], double& dmax2) {
  const unsigned lane = threadIdx.x & 31;
  const double qscale = 4294967295.0 / r2;          // quantised key: monotone non-decreasing in d^2, < 2^32 for d^2 < r^2
  const double4* __restrict__ P = reinterpret_cast<const double4*>(S.phPos); const double4* __restrict__ W = reinterpret_cast<const double4*>(S.phPwr);
  // F(j, d2, q, ok) warp-wide for every candidate, ok = d2 < r2.  The per-range walk gives each lane the same photons in the same order on
  // every level and in the final pass.
  auto each = [&](auto&& F) {
    phEachRange(sh, R, [&](uint32_t j, bool ok) {
      double d2 = 0;
      if (ok) { const double4 q = P[j]; const double dx = p.x - q.x, dy = p.y - q.y, dz = p.z - q.z; d2 = dx * dx + dy * dy + dz * dz; ok = d2 < r2; }
      F(j, d2, ok ? (uint32_t)(d2 * qscale) : 0u, ok);
    });
  };
  // level loop: keys with (q >> shift) < prefix are already known to be inside; those == prefix are undecided
  uint32_t prefix = 0; int shift = 32; int need = S.g.kNhood; bool takeAllUndecided = false, haveList = false;
  while (true) {
    const int nshift = shift - 8;
    __syncwarp();
    for (int i = lane; i < DRT_PH_BINS; i += 32) sh.hist[i] = 0;
    __syncwarp();
    unsigned m = 0;
    each([&](uint32_t, double, uint32_t q, bool ok) {
      const bool und = ok && (shift == 32 || (q >> shift) == prefix);
      if (und) atomicAdd(&sh.hist[(q >> nshift) & 255u], 1u);
      m += __popc(__ballot_sync(0xffffffffu, und));
    });
    __syncwarp();
    if (needAll && shift == 32 && (int)m < need) return false;              // the guessed radius holds fewer than k photons: caller retries with the full one
    if ((int)m <= need) { takeAllUndecided = true; break; }                 // fewer undecided candidates than still needed: all of them are in
    uint32_t binSel, before, inBin; phFindBin(sh, (uint32_t)need, binSel, before, inBin);
    need -= (int)before; prefix = (shift == 32) ? binSel : ((prefix << 8) | binSel); shift = nshift;
    if (inBin <= DRT_PH_LIST) { haveList = true; break; }
    if (shift == 0) break;                                                    // > DRT_PH_LIST photons with identical 32-bit distance keys: take by index order below
  }
  // final pass: accumulate everything decided-in; collect the boundary bin
  if (lane == 0) sh.listN = 0;
  __syncwarp();
  double s0 = 0, s1 = 0, s2 = 0, mx = 0; int tieTaken = 0;
  each([&](uint32_t j, double d2, uint32_t q, bool ok) {
    bool in = false, bnd = false;
    if (ok) {
      if (takeAllUndecided) in = (shift == 32) || ((q >> shift) <= prefix);
      else { const uint32_t hb = q >> shift; in = hb < prefix; bnd = hb == prefix; }
    }
    const unsigned bm = __ballot_sync(0xffffffffu, bnd);
    if (haveList) {
      if (bnd) { const uint32_t at = sh.listN + __popc(bm & ((1u << lane) - 1u)); if (at < DRT_PH_LIST) { sh.listD2[at] = d2; sh.listIdx[at] = j; } }
      __syncwarp();
      if (lane == 0) sh.listN += __popc(bm);
      __syncwarp();
    } else if (bm) {          // degenerate ties (> DRT_PH_LIST equal 32-bit keys): first `need` in index order
      if (bnd) in = (tieTaken + __popc(bm & ((1u << lane) - 1u))) < need;
      tieTaken += __popc(bm);
    }
    if (in) { const double4 w = W[j]; s0 += w.x; s1 += w.y; s2 += w.z; mx = fmax(mx, d2); }
  });
  if (haveList) phRankList(sh, need, W, s0, s1, s2, mx);
  phWarpSum(s0, s1, s2, mx, sum, dmax2);
  return true;
}

// FP32 pre-test selection: the same exact result from ONE histogram pass and one collection pass, both in FP32.
// The FP64 selection re-reads every candidate's 32-byte position and re-forms d^2 in FP64 for every radix level (2-3 walks of ~11 FP64-pipe
// operations per candidate: the half-rate FP64 pipe is what bounds dense maps).  Here d^2 is formed in FP32 from a float4 mirror of the positions;
// with u = 2^-24, A = largest |coordinate| of a photon and rho = sqrt(r2),
//     |d2_32 - d2| <= delta = 2 sqrt(3) rho e + 3 e^2 + 4 u r2,     e = u (|p|_inf + A + rho)        (coordinate rounding + one rounding per operation)
// for every candidate with d2 <= r2.  256 bins of width w = r2/256 over the FP32 values; the method is used only if 4 delta < w.  Then, with b the
// bin where the running count reaches k: every candidate binned <= b-2 is among the k nearest (the k-th true distance is >= edge(b) - delta),
// every candidate binned >= b+2 is not, and the <= 128 candidates of bins b-1..b+1 are resolved exactly -- FP64 d^2 from the FP64 positions,
// (d^2, index) order -- by the same boundary-list ranking as the FP64 selection.  The k-th neighbour itself is always in that list, so the d^2
// that leaves the function is the FP64 value.  Candidates within delta of the radius are classified by their FP64 d^2.  Returns 1 (done), 0
// (needAll and fewer than k photons inside r2) or -1 (margin too wide, or a boundary list longer than 128: the FP64 selection decides).
__device__ inline int phWarpGather32(const DScene& S, D3 p, double r2, bool needAll, PhRanges R, PhWarpShared& sh, double sum[3], double& dmax2) {
  const unsigned lane = threadIdx.x & 31; const int K = S.g.kNhood;
  const float u = 5.9604644775390625e-8f, rho = __double2float_ru(sqrt(r2)), r2f = __double2float_ru(r2);
  const float pm = fmaxf(fmaxf(fabsf(__double2float_ru(fabs(p.x))), fabsf(__double2float_ru(fabs(p.y)))), fabsf(__double2float_ru(fabs(p.z))));
  const float e = 1.01f * u * (pm + S.phAbsMax + rho), delta = 1.05f * (3.4641016f * rho * e + 3.0f * e * e + 4.0f * u * r2f);
  if (!(4.0f * delta < r2f * (1.0f / 256.0f)) || !(r2f < 1e30f) || !(r2f > 1e-30f)) return -1;
  const float rIn = __double2float_rd(r2) - delta, rOut = r2f + delta, scale = 256.0f / r2f, px = (float)p.x, py = (float)p.y, pz = (float)p.z;
  const float4* __restrict__ P32 = reinterpret_cast<const float4*>(S.phPos32);
  const double4* __restrict__ P = reinterpret_cast<const double4*>(S.phPos); const double4* __restrict__ W = reinterpret_cast<const double4*>(S.phPwr);
  auto exactD2 = [&](uint32_t j) { const double4 q = P[j]; const double dx = p.x - q.x, dy = p.y - q.y, dz = p.z - q.z; return dx * dx + dy * dy + dz * dz; };
  // bin of candidate j, or -1 when it is outside the radius
  auto binOf = [&](uint32_t j) -> int {
    const float4 q = P32[j]; const float dx = px - q.x, dy = py - q.y, dz = pz - q.z; const float d2 = fmaf(dz, dz, fmaf(dy, dy, dx * dx));
    if (d2 > rOut) return -1;
    if (d2 >= rIn && !(exactD2(j) < r2)) return -1;
    const int b = (int)(d2 * scale); return b > 255 ? 255 : b;
  };
  for (int i = lane; i < DRT_PH_BINS; i += 32) sh.hist[i] = 0;
  if (lane == 0) sh.listN = 0;
  __syncwarp();
  unsigned m = 0;
  phEachFlat(sh, R, [&](uint32_t j, bool valid) { const int bin = valid ? binOf(j) : -1; if (bin >= 0) atomicAdd(&sh.hist[bin], 1u); m += __popc(__ballot_sync(0xffffffffu, bin >= 0)); });
  __syncwarp();
  if (needAll && (int)m < K) return 0;
  if (m == 0) return 1;
  // boundary bin b: running count reaches k (m > k), or the highest non-empty bin (m <= k: every photon inside r2 is taken)
  const uint32_t target = (int)m > K ? (uint32_t)K : m;
  uint32_t bSel, before, inBin; phFindBin(sh, target, bSel, before, inBin);
  const uint32_t prev = bSel > 0 ? sh.hist[bSel - 1] : 0u, next = bSel < DRT_PH_BINS - 1 ? sh.hist[bSel + 1] : 0u;
  if (prev + inBin + next > DRT_PH_LIST) return -1;
  const int bLo = (int)bSel - 1, bHi = (int)bSel + 1;        // exact zone; bins < bLo are in, bins > bHi are out
  const int need = (int)target - (int)(before - prev);       // >= 1: the running count through bin b-1 is below the target
  double s0 = 0, s1 = 0, s2 = 0, mx = 0;
  phEachFlat(sh, R, [&](uint32_t j, bool valid) {
    const int bin = valid ? binOf(j) : -1;
    if (bin >= 0 && bin < bLo) { const double4 w = W[j]; s0 += w.x; s1 += w.y; s2 += w.z; }
    const bool bnd = bin >= bLo && bin <= bHi; const unsigned bm = __ballot_sync(0xffffffffu, bnd);
    if (bm) {
      if (bnd) { const uint32_t at = sh.listN + __popc(bm & ((1u << lane) - 1u)); sh.listD2[at] = exactD2(j); sh.listIdx[at] = j; }
      __syncwarp();
      if (lane == 0) sh.listN += __popc(bm);
      __syncwarp();
    }
  });
  phRankList(sh, need, W, s0, s1, s2, mx);
  phWarpSum(s0, s1, s2, mx, sum, dmax2);
  return 1;
}

// One search of the warp tier over the cells lo..hi (coarse rows, or the fine cells of a plan): one candidate list, the FP32 selection, and
// the FP64 one when the FP32 one cannot decide.  False when `needAll` and fewer than k photons lie inside r2.
__device__ inline bool phWarpGather(const DScene& S, D3 p, double r2, bool needAll, bool fine, const int lo[3], const int hi[3], PhWarpShared& sh, double sum[3], double& dmax2) {
  sum[0] = sum[1] = sum[2] = 0; dmax2 = 0;
  const PhRanges R = phWarpRanges(S, fine, lo, hi, sh);
  const int g = phWarpGather32(S, p, r2, needAll, R, sh, sum, dmax2);
  return g < 0 ? phWarpGather64(S, p, r2, needAll, R, sh, sum, dmax2) : g > 0;
}

// cheap per-lane test: does any cell the search sphere's bounding cube overlaps hold a photon at all?  (sparse caustic maps: most queries do not)
__device__ inline uint32_t phCountCandidates(const DScene& S, const int lo[3], const int hi[3]) {
  uint32_t c = 0;
  for (int cz = lo[2]; cz <= hi[2]; ++cz) for (int cy = lo[1]; cy <= hi[1]; ++cy) {
    uint32_t a, b; phRowRange(S, false, cy, cz, lo[0], hi[0], a, b); c += b - a;
  }
  return c;
}
// Dense neighbourhoods: the k-th neighbour is far closer than r, so most of the r-sphere's candidates are wasted work.  Per query (lane-parallel):
//   count the photons in the fine cube of half-width 1, 2, 3 around p's fine cell; the first one expected to hold >= 1.25 k photons inside its
//   inscribed search sphere gives the plan
//   "search radius s * fineCell over that cube" -- exact if >= k photons turn out to lie inside that radius (every photon closer than s fine
//   cells to p is in the cube), otherwise the caller falls back to the full radius over the coarse rows.
struct PhPlan { int fineHalf; int c[3]; int h[3]; double r2; int f[3]; double r2max; bool shrunk; };      // fineHalf < 0: coarse rows c..h, else fine cells c..h with threshold r2; f / r2max: the un-shrunk plan (cube f +- fineHalf, radius of fineHalf fine cells)
__device__ __forceinline__ uint32_t phCountFineCube(const DScene& S, const int f[3], int s) {
  const int fdx = 4 * (int)S.gridDim[0], fdy = 4 * (int)S.gridDim[1], fdz = 4 * (int)S.gridDim[2];
  const int z0 = max(f[2] - s, 0), z1 = min(f[2] + s, fdz - 1), y0 = max(f[1] - s, 0), y1 = min(f[1] + s, fdy - 1), x0 = max(f[0] - s, 0), x1 = min(f[0] + s, fdx - 1);
  uint32_t c = 0;
  for (int fz = z0; fz <= z1; ++fz) for (int fy = y0; fy <= y1; ++fy)
    for (int fx = x0; fx <= x1; ) { const int runEnd = min(x1, fx | 3); uint32_t a, b; phRowRange(S, true, fy, fz, fx, runEnd, a, b); c += b - a; fx = runEnd + 1; }
  return c;
}
// The plan: a search radius rho <= s fine cells (s = 1, 2, 3) and the block of fine cells its sphere's bounding cube overlaps.  s = the first
// half-width whose cube is expected to hold >= 1.25 k photons inside its inscribed sphere (surface distribution: share pi s^2 / (2s+1)^2); rho is
// then shrunk from s fine cells to the radius expected to hold 1.5 k photons under the same area scaling -- the scanned block shrinks with it,
// from (2s+1)^3 cells to the cells [p - rho, p + rho] touches.  Exact whatever the estimate: a plan's result is used only if >= k photons turn
// out to lie inside rho (then the k nearest are among them, and every photon inside rho is in a scanned cell); otherwise the caller searches the
// full radius over the coarse rows.
__device__ __forceinline__ void phMakePlan(const DScene& S, D3 p, uint32_t coarseCount, const int lo[3], const int hi[3], PhPlan& pl) {
  const int K = S.g.kNhood; pl.fineHalf = -1; pl.r2 = S.g.phMaxDist2; pl.r2max = pl.r2; pl.shrunk = false;
  for (int k = 0; k < 3; ++k) { pl.c[k] = lo[k]; pl.h[k] = hi[k]; pl.f[k] = 0; }
  if (coarseCount < (uint32_t)(8 * K)) return;
  const double cf = S.cellSize * 0.25, pp[3] = {p.x, p.y, p.z}; int f[3]; bool inside = true;
  for (int k = 0; k < 3; ++k) { const double a = floor((pp[k] - S.gridMin[k]) / cf); const int fd = 4 * (int)S.gridDim[k]; if (!(a >= 0) || !(a <= fd - 1)) inside = false; f[k] = (int)a; }
  if (!inside) return;
  const double frac[4] = {0.0, 0.349, 0.503, 0.577};
  for (int s = 1; s <= 3; ++s) {
    const double radMax = s * cf * (1.0 - 1e-6);                               // 1e-6: a photon's own fine index is a rounded quotient
    if (!(radMax * radMax <= S.g.phMaxDist2)) return;                          // never search beyond the scene's radius (find_near requires d^2 < r^2): when the
                                                                               // grid had to double its cell size the fine cells are wider than r/4 and the plan does not apply
    const double inSphere = (double)phCountFineCube(S, f, s) * frac[s];
    if (inSphere >= 1.25 * K) {
      double rad = radMax * sqrt(1.5 * K / inSphere); if (!(rad < radMax)) rad = radMax;
      const double reach = rad * (1.0 + 1e-6) + 1e-9 * cf;                     // cells the sphere can touch, with room for the rounding of a photon's own cell index
      pl.fineHalf = s; pl.r2 = rad * rad; pl.r2max = radMax * radMax; pl.shrunk = rad < radMax;
      for (int k = 0; k < 3; ++k) { const int fd = 4 * (int)S.gridDim[k]; const int a = (int)floor((pp[k] - reach - S.gridMin[k]) / cf), b = (int)floor((pp[k] + reach - S.gridMin[k]) / cf);
        pl.c[k] = max(max(a, f[k] - s), 0); pl.h[k] = min(min(b, f[k] + s), fd - 1); pl.f[k] = f[k]; }
      return;
    }
  }
}
// ---- one query per lane, three tiers by the number of photons in the candidate cells (all exact):
//   <= k              the lane sums its candidates itself (nothing to select)
//   <= DRT_PH_LANE_MAX the lane runs a two-pass histogram selection itself (neighbouring lanes read the same photons: mostly uniform loads)
//   larger            the warp serves the query cooperatively (phWarpGather), over a fine cube first when the neighbourhood is dense
// Results per lane: sum of the k nearest powers and d^2 of the farthest (0 = no photon in range). `path` (optional) reports the tier taken.
struct PhLaneShared { uint16_t laneHist[128 * 128]; };      // lane-private 128-bin histograms laid out [bin][thread]
struct PhWarpTierShared { PhWarpShared warp[4]; };
// tiers 1 and 2; returns true when the query is left for the warp-cooperative tier
__device__ inline bool phLaneTiers(const DScene& S, bool needs, D3 loc, PhLaneShared& sm, double sum[3], double& dmax2, int* path) {
  const double r2 = S.g.phMaxDist2; const int K = S.g.kNhood;
  sum[0] = sum[1] = sum[2] = 0; dmax2 = 0; if (path) *path = 0;
  bool few = false; int lo[3] = {0, 0, 0}, hi[3] = {0, 0, 0};
  needs = needs && S.numPhotons > 0 && K > 0;
  if (needs) {
    needs = phCellRange(S, loc, r2, lo, hi); const uint32_t cnt = needs ? phCountCandidates(S, lo, hi) : 0u; needs = cnt > 0; few = cnt <= (uint32_t)K;
    const double4* __restrict__ P = reinterpret_cast<const double4*>(S.phPos); const double4* __restrict__ W = reinterpret_cast<const double4*>(S.phPwr);
    if (needs && few) {                                                    // tier 1. Sum order = photon order in the sorted array
      double s0 = 0, s1 = 0, s2 = 0, mx = 0;
      for (int cz = lo[2]; cz <= hi[2]; ++cz) for (int cy = lo[1]; cy <= hi[1]; ++cy) {
        uint32_t a, b; phRowRange(S, false, cy, cz, lo[0], hi[0], a, b);
        for (uint32_t j = a; j < b; ++j) { const double4 q = P[j]; const double dx = loc.x - q.x, dy = loc.y - q.y, dz = loc.z - q.z, d2 = dx * dx + dy * dy + dz * dz;
          if (d2 < r2) { const double4 w = W[j]; s0 += w.x; s1 += w.y; s2 += w.z; mx = fmax(mx, d2); } }
      }
      sum[0] = s0; sum[1] = s1; sum[2] = s2; dmax2 = mx; needs = false; if (path) *path = 1;
    }
    if (needs && cnt <= DRT_PH_LANE_MAX) {                                 // tier 2 (an FP32 pre-test form of this tier was measured and lost: profiles/r2_tuning.md)
      // pass 1 bins d^2 into the lane's histogram (bin index monotone in d^2) and finds the bin of the k-th neighbour; pass 2 sums the bins
      // below it and resolves the boundary bin exactly from a register list sorted by (d^2, index). A boundary bin with more than 8 photons
      // hands the query to the warp-cooperative tier.
      const double bscale = 127.99999 / r2; uint16_t* h = sm.laneHist + threadIdx.x;
      for (int b = 0; b < 128; ++b) h[b * 128] = 0;
      int m = 0;
      for (int cz = lo[2]; cz <= hi[2]; ++cz) for (int cy = lo[1]; cy <= hi[1]; ++cy) {
        uint32_t a, b; phRowRange(S, false, cy, cz, lo[0], hi[0], a, b);
        for (uint32_t j = a; j < b; ++j) { const double4 q = P[j]; const double dx = loc.x - q.x, dy = loc.y - q.y, dz = loc.z - q.z, d2 = dx * dx + dy * dy + dz * dz;
          if (d2 < r2) { ++m; ++h[(int)(d2 * bscale) * 128]; } }
      }
      if (m == 0) { needs = false; if (path) *path = 2; }
      else {
        int bsel = 128, below = 0;
        if (m > K) { int c = 0; for (int b = 0; b < 128; ++b) { const int hb = h[b * 128]; if (c + hb >= K) { bsel = b; below = c; break; } c += hb; } }
        const int need = K - below;                                       // photons to take from the boundary bin (m > K only)
        double s0 = 0, s1 = 0, s2 = 0, mx = 0, ld[8]; uint32_t lj[8]; int ln = 0; bool overflow = false;
        for (int cz = lo[2]; cz <= hi[2]; ++cz) for (int cy = lo[1]; cy <= hi[1]; ++cy) {
          uint32_t a, b; phRowRange(S, false, cy, cz, lo[0], hi[0], a, b);
          for (uint32_t j = a; j < b; ++j) { const double4 q = P[j]; const double dx = loc.x - q.x, dy = loc.y - q.y, dz = loc.z - q.z, d2 = dx * dx + dy * dy + dz * dz;
            if (d2 < r2) { const int bin = (int)(d2 * bscale);
              if (bin < bsel) { const double4 w = W[j]; s0 += w.x; s1 += w.y; s2 += w.z; mx = fmax(mx, d2); }
              else if (bin == bsel) {
                if (ln == 8) overflow = true;
                else { int pos = ln; while (pos > 0 && (ld[pos - 1] > d2)) { ld[pos] = ld[pos - 1]; lj[pos] = lj[pos - 1]; --pos; } ld[pos] = d2; lj[pos] = j; ++ln; } } } }
        }
        if (!overflow) {
          for (int t = 0; t < need && t < ln; ++t) { const double4 w = W[lj[t]]; s0 += w.x; s1 += w.y; s2 += w.z; mx = fmax(mx, ld[t]); }
          sum[0] = s0; sum[1] = s1; sum[2] = s2; dmax2 = mx; needs = false; if (path) *path = 2;
        }
      }
    }
  }
  return needs;
}
// tier 3 / 4: the warp serves its pending queries one at a time
__device__ inline void phWarpTier(const DScene& S, bool pending, D3 loc, PhWarpTierShared& sm, double sum[3], double& dmax2, int* path) {
  const unsigned lane = threadIdx.x & 31; const double r2 = S.g.phMaxDist2; const int K = S.g.kNhood;
  int lo[3] = {0, 0, 0}, hi[3] = {0, 0, 0}; PhPlan pl; pl.fineHalf = -1; pl.r2 = r2; pl.r2max = r2; pl.shrunk = false; for (int k = 0; k < 3; ++k) pl.c[k] = pl.h[k] = pl.f[k] = 0;
  bool needs = pending && S.numPhotons > 0 && K > 0;
  if (needs) { needs = phCellRange(S, loc, r2, lo, hi); const uint32_t cnt = needs ? phCountCandidates(S, lo, hi) : 0u; needs = cnt > 0; if (needs) phMakePlan(S, loc, cnt, lo, hi, pl); }
  PhWarpShared& sh = sm.warp[threadIdx.x >> 5];
  unsigned mask = __ballot_sync(0xffffffffu, needs);
  while (mask) {
    const int src = __ffs(mask) - 1; mask &= mask - 1;
    const D3 p = d3(__shfl_sync(0xffffffffu, loc.x, src), __shfl_sync(0xffffffffu, loc.y, src), __shfl_sync(0xffffffffu, loc.z, src));
    const int fineHalf = __shfl_sync(0xffffffffu, pl.fineHalf, src);
    int qlo[3], qhi[3]; double qs[3], qd; bool done = false;
    if (fineHalf > 0) {
      const double pr2 = __shfl_sync(0xffffffffu, pl.r2, src);
#pragma unroll
      for (int k = 0; k < 3; ++k) { qlo[k] = __shfl_sync(0xffffffffu, pl.c[k], src); qhi[k] = __shfl_sync(0xffffffffu, pl.h[k], src); }
      done = phWarpGather(S, p, pr2, true, true, qlo, qhi, sh, qs, qd);
      if (!done && __shfl_sync(0xffffffffu, (int)pl.shrunk, src) != 0) {      // fewer than k photons inside the shrunk radius: the plan's full radius over its whole cube, before the coarse rows
        const double pr2m = __shfl_sync(0xffffffffu, pl.r2max, src);
#pragma unroll
        for (int k = 0; k < 3; ++k) { const int fk = __shfl_sync(0xffffffffu, pl.f[k], src); qlo[k] = max(fk - fineHalf, 0); qhi[k] = min(fk + fineHalf, 4 * (int)S.gridDim[k] - 1); }
        done = phWarpGather(S, p, pr2m, true, true, qlo, qhi, sh, qs, qd);
      }
    }
    if (!done) {
#pragma unroll
      for (int k = 0; k < 3; ++k) { qlo[k] = __shfl_sync(0xffffffffu, lo[k], src); qhi[k] = __shfl_sync(0xffffffffu, hi[k], src); }
      phWarpGather(S, p, r2, false, false, qlo, qhi, sh, qs, qd);
    }
    if ((int)lane == src) { sum[0] = qs[0]; sum[1] = qs[1]; sum[2] = qs[2]; dmax2 = qd; if (path) *path = done ? 4 : 3; }
    __syncwarp();
  }
}

// Run between k_shade (local = ambient) and k_light (local += direct), which is the reference's accumulation order (myObjShader.java:413-425).
// Two kernels so that the warp-cooperative tier keeps its occupancy (96 registers, 16 KB shared) and the lane tiers their histogram space:
// k_photon_gather_lane resolves tiers 1-2 and marks what is left in SurfRec::pad, k_photon_gather_warp serves the marked queries.
__device__ __forceinline__ void phApply(const DScene& S, int shIdx, const double sum[3], double dmax2, double* l) {
  if (!(dmax2 > 0)) return;
  const double area = DRT_PI_F * dmax2; const D3 irr = d3(sum[0] / area, sum[1] / area, sum[2] / area); const FShader& sh = S.shaders[shIdx];
  if (sh.flags & SF_IS_CAUSTIC_PHTN) { l[0] = l[0] + irr.x; l[1] = l[1] + irr.y; l[2] = l[2] + irr.z; }
  else { l[0] = l[0] + sh.diff[0] * irr.x; l[1] = l[1] + sh.diff[1] * irr.y; l[2] = l[2] + sh.diff[2] * irr.z; }
}
__global__ void __launch_bounds__(128) k_photon_gather_lane(const __grid_constant__ DScene S, Wave w, SurfRec* __restrict__ surf, NodeRec* __restrict__ nodesBase, const Counters* ctr) {
  __shared__ PhLaneShared sm;
  const long long n = waveCount(w, ctr); NodeRec* __restrict__ nodes = nodesBase + ((w.level == 0) ? 0 : waveNodeOffset(w, ctr, w.level));
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const SurfRec s = surf[i]; if (!s.valid) continue;
    const FShader& sh = S.shaders[s.shader];
    const bool needs = !(sh.flags & SF_SIMPLE) && (sh.KRefl == 0.0) && (sh.flags & SF_USE_PHOTON);
    double sum[3], dmax2; const bool pending = phLaneTiers(S, needs, d3(s.loc[0], s.loc[1], s.loc[2]), sm, sum, dmax2, nullptr);
    surf[i].pad = pending ? 1 : 0;
    if (needs && !pending) phApply(S, s.shader, sum, dmax2, nodes[i].local);
  }
}
__global__ void __launch_bounds__(128) k_photon_gather_warp(const __grid_constant__ DScene S, Wave w, const SurfRec* __restrict__ surf, NodeRec* __restrict__ nodesBase, const Counters* ctr) {
  __shared__ PhWarpTierShared sm;
  const long long n = waveCount(w, ctr); NodeRec* __restrict__ nodes = nodesBase + ((w.level == 0) ? 0 : waveNodeOffset(w, ctr, w.level));
  for (long long base = (long long)blockIdx.x * blockDim.x; base < n; base += (long long)gridDim.x * blockDim.x) {
    const long long i = base + threadIdx.x;
    bool pending = false; D3 loc = d3(0, 0, 0); int shIdx = -1;
    if (i < n) { pending = surf[i].valid && surf[i].pad == 1; if (pending) { shIdx = surf[i].shader; loc = d3(surf[i].loc[0], surf[i].loc[1], surf[i].loc[2]); } }
    if (!__any_sync(0xffffffffu, pending)) continue;
    double sum[3], dmax2; phWarpTier(S, pending, loc, sm, sum, dmax2, nullptr);
    if (pending) phApply(S, shIdx, sum, dmax2, nodes[i].local);
  }
}

// parity probe: the same routines at explicit points, one lane per point: out = {sum r,g,b, dmax2, tier taken}
__global__ void __launch_bounds__(128) k_photon_probe(const __grid_constant__ DScene S, long long n, const double* __restrict__ pts, double* __restrict__ out) {
  __shared__ union ProbeShared { PhLaneShared sl; PhWarpTierShared sw; } u;       // the two tiers run one after the other (48 KB static limit)
  const long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; const bool ok = q < n;
  const D3 p = ok ? d3(pts[3 * q], pts[3 * q + 1], pts[3 * q + 2]) : d3(0, 0, 0);
  double sum[3], dmax2; int path = 0;
  const bool pending = phLaneTiers(S, ok, p, u.sl, sum, dmax2, &path);
  __syncthreads();
  double s2[3], d2; int path2 = 0; phWarpTier(S, pending, p, u.sw, s2, d2, &path2);
  if (pending) { sum[0] = s2[0]; sum[1] = s2[1]; sum[2] = s2[2]; dmax2 = d2; path = path2; }
  if (ok) { out[5 * q] = sum[0]; out[5 * q + 1] = sum[1]; out[5 * q + 2] = sum[2]; out[5 * q + 3] = dmax2; out[5 * q + 4] = (double)path; }
}

// ---------------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------------
struct PhotonMap {
  bool built = false, emitted = false; unsigned long long count = 0, segments = 0;
  DBuf<PhotonRec> rec;                                          // canonical-order records (emission output / grid input)
  DBuf<double4> pos, pwr; DBuf<float4> pos32; DBuf<uint32_t> cellStart;      // the sorted map
  PhGrid grid{}; float msEmit = 0, msBuild = 0;
  DBuf<PhotonRec> sSlots; DBuf<uint32_t> sCnt, sOff, sScan, sKeys[2], sVals[2], sHist; DBuf<double> sBounds; DEvent evA, evB;

  void reset() { built = false; emitted = false; count = 0; segments = 0; }

  // photons [i0, i1) of every light -> appended to `rec` in canonical order. Chunked so the slot buffer stays bounded.
  void emitRange(const DScene& ds, long long i0, long long i1, Counters* ctr, Counters* ctrHost, cudaStream_t st) {
    built = false; emitted = true; count = 0; segments = 0;
    const int nl = ds.g.numLights; if (nl <= 0 || i1 <= i0 || ds.g.photonKind == 0) return;
    const int maxStore = ds.g.photonKind == 1 ? 1 : (ds.g.numPhotonRays + 1);
    const long long chunkPhotons = std::max<long long>(1, (1ll << 21) / nl);
    const long long maxThreads = std::min(chunkPhotons, i1 - i0) * nl;
    PhotonRec* slots = sSlots.ensure((size_t)maxThreads * maxStore, st); uint32_t* cnt = sCnt.ensure((size_t)maxThreads + 1, st); uint32_t* off = sOff.ensure((size_t)maxThreads + 1, st);
    uint32_t* scratch = sScan.ensure((size_t)scanScratchWords(maxThreads + 1), st);
    CK(cudaEventRecord(evA, st));
    CK(cudaMemsetAsync(&ctr->pad, 0, sizeof(unsigned long long), st));
    for (long long c0 = i0; c0 < i1; c0 += chunkPhotons) {
      const long long np = std::min(chunkPhotons, i1 - c0), nt = np * nl;
      CK(cudaMemsetAsync(cnt + nt, 0, 4, st));
      k_photon_emit<<<(unsigned)((nt + 127) / 128), 128, 0, st>>>(ds, c0, nt, maxStore, slots, cnt, ctr); ++g_kernelLaunches;
      scanExclusiveU32(cnt, off, nt + 1, scratch, st);
      uint32_t total = 0; CK(cudaMemcpyAsync(&total, off + nt, 4, cudaMemcpyDeviceToHost, st)); CK(cudaStreamSynchronize(st));
      rec.ensure(count + total, st, true);
      if (total) { k_photon_compact<<<(unsigned)((nt + 255) / 256), 256, 0, st>>>(nt, maxStore, slots, cnt, off, rec.p + count); ++g_kernelLaunches; }
      count += total;
    }
    CK(cudaMemcpyAsync(ctrHost, ctr, sizeof(Counters), cudaMemcpyDeviceToHost, st));
    CK(cudaEventRecord(evB, st)); CK(cudaStreamSynchronize(st)); CK(cudaGetLastError());
    segments = ctrHost->pad; CK(cudaEventElapsedTime(&msEmit, evA, evB));
  }
  // replace the record store with `n` records that already live on the device (multi-GPU: the all-gathered set)
  void setRecords(const PhotonRec* srcDev, unsigned long long n, cudaStream_t st) {
    built = false; emitted = true; count = 0; rec.ensure((size_t)n, st);
    if (n) CK(cudaMemcpyAsync(rec.p, srcDev, n * sizeof(PhotonRec), cudaMemcpyDeviceToDevice, st));
    count = n; CK(cudaStreamSynchronize(st));
  }

  void buildGrid(DScene& ds, cudaStream_t st) {
    ds.numPhotons = 0; ds.phPos = nullptr; ds.phPwr = nullptr; ds.cellStart = nullptr; ds.phPos32 = nullptr; ds.phAbsMax = 0; ds.padP = 0; built = true; msBuild = 0;
    if (count == 0) return;
    if (count >= 0xFFFFFFF0ull) throw std::runtime_error("photon map larger than 2^32 records");
    CK(cudaEventRecord(evA, st));
    const long long n = (long long)count;
    // bounds
    const int nbB = 592; double* bmm = sBounds.ensure((size_t)nbB * 6, st);
    k_photon_bounds<<<nbB, 256, 0, st>>>(rec.p, n, bmm); ++g_kernelLaunches;
    std::vector<double> hb(nbB * 6); CK(cudaMemcpyAsync(hb.data(), bmm, hb.size() * 8, cudaMemcpyDeviceToHost, st)); CK(cudaStreamSynchronize(st));
    double mn[3] = {DRT_DMAX, DRT_DMAX, DRT_DMAX}, mx[3] = {-DRT_DMAX, -DRT_DMAX, -DRT_DMAX};
    for (int b = 0; b < nbB; ++b) for (int k = 0; k < 3; ++k) { mn[k] = std::min(mn[k], hb[b * 6 + k]); mx[k] = std::max(mx[k], hb[b * 6 + 3 + k]); }
    double cell = std::sqrt(ds.g.phMaxDist2); if (!(cell > 0)) cell = 1e-3;
    PhGrid G;
    while (true) {
      double cells = 1; for (int k = 0; k < 3; ++k) { double d = std::floor((mx[k] - mn[k]) / cell) + 1; if (d < 1) d = 1; G.dim[k] = (uint32_t)std::min(d, 4.0e9); cells *= d; }
      if (cells <= (double)(1u << 22)) break;          // x 64 fine sub-cells = at most 2^28 cellStart entries (1 GiB)
      cell *= 2;
    }
    G.cell = cell; for (int k = 0; k < 3; ++k) G.gmin[k] = mn[k]; G.nCells = G.dim[0] * G.dim[1] * G.dim[2] * 64u; grid = G;     // nCells counts FINE cells
    // keys + per-cell counts, cellStart = exclusive scan (nCells + 1 entries: cellStart[nCells] = n)
    uint32_t* cells = cellStart.ensure((size_t)G.nCells + 1, st); pos.ensure((size_t)n, st); pwr.ensure((size_t)n, st); pos32.ensure((size_t)n, st);
    uint32_t *keys[2], *vals[2]; const long long nb = radixBlocks(n);
    for (int k = 0; k < 2; ++k) { keys[k] = sKeys[k].ensure((size_t)n, st); vals[k] = sVals[k].ensure((size_t)n, st); }
    const long long scanWords = std::max(scanScratchWords(256 * nb), scanScratchWords((long long)G.nCells + 1));
    uint32_t* hist = sHist.ensure((size_t)256 * nb, st); uint32_t* scratch = sScan.ensure((size_t)scanWords, st);
    CK(cudaMemsetAsync(cells, 0, ((size_t)G.nCells + 1) * 4, st));
    k_photon_cellkeys<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(rec.p, n, G, keys[0], cells); ++g_kernelLaunches;
    scanExclusiveU32(cells, cells, (long long)G.nCells + 1, scratch, st);
    int bits = 1; while ((1ull << bits) < (unsigned long long)G.nCells) ++bits;
    const int cur = radixSortPairs(keys, vals, n, bits, true, hist, scratch, st);
    k_photon_reorder<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(rec.p, vals[cur], n, pos.p, pwr.p, pos32.p); ++g_kernelLaunches;
    CK(cudaEventRecord(evB, st)); CK(cudaStreamSynchronize(st)); CK(cudaGetLastError()); CK(cudaEventElapsedTime(&msBuild, evA, evB));
    ds.numPhotons = (uint32_t)n; ds.phPos = reinterpret_cast<const double*>(pos.p); ds.phPwr = reinterpret_cast<const double*>(pwr.p); ds.cellStart = cells; ds.phPos32 = reinterpret_cast<const float*>(pos32.p);
    { double a = 0; for (int k = 0; k < 3; ++k) a = std::max(a, std::max(std::fabs(mn[k]), std::fabs(mx[k]))); const float f = (float)a; ds.phAbsMax = f >= a ? f : std::nextafter(f, INFINITY); ds.padP = 0; }
    for (int k = 0; k < 3; ++k) { ds.gridDim[k] = G.dim[k]; ds.gridMin[k] = G.gmin[k]; } ds.cellSize = G.cell;
  }

  void emitAndBuild(DScene& ds, Counters* ctr, Counters* ctrHost, cudaStream_t st) { emitRange(ds, 0, ds.g.numPhotonsCast, ctr, ctrHost, st); buildGrid(ds, st); }

  long long download(double* out6, long long cap, cudaStream_t st) {
    long long n = std::min<long long>((long long)count, cap); if (n <= 0 || !out6) return (long long)count;
    CK(cudaMemcpyAsync(out6, rec.p, (size_t)n * sizeof(PhotonRec), cudaMemcpyDeviceToHost, st)); CK(cudaStreamSynchronize(st)); return n;
  }
};

}  // namespace drt
