// Device-side double-precision helpers and the counter-based sampler.
// The translation unit is compiled with -fmad=false: the reference (Java, strict IEEE, no FMA contraction)
// defines the bits of every comparison that decides a hit, so multiply-add is never fused here.
// Operation order follows myVector.java:27-43 (vector), :85-90 (matrix x vertex).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "scene_flat.h"

namespace drt {

#define DRT_EPS .0000001
#define DRT_DMAX 1.7976931348623157e308
#define DRT_PI 3.141592653589793
#define DRT_PI_F 3.1415927410125732        // (double)(float)pi
#define DRT_TWO_PI_F 6.2831854820251465    // (double)(float)(2 pi)

struct D3 { double x, y, z; };
__device__ __forceinline__ D3 d3(double x, double y, double z) { D3 r; r.x = x; r.y = y; r.z = z; return r; }
__device__ __forceinline__ double dot3(D3 a, D3 b) { return ((a.x * b.x) + (a.y * b.y) + (a.z * b.z)); }
__device__ __forceinline__ D3 cross3(D3 a, D3 b) { return d3((a.y * b.z) - (a.z * b.y), (a.z * b.x) - (a.x * b.z), (a.x * b.y) - (a.y * b.x)); }
__device__ __forceinline__ double mag3(D3 a) { return sqrt(((a.x * a.x) + (a.y * a.y) + (a.z * a.z))); }
__device__ __forceinline__ D3 norm3(D3 a) { double m = mag3(a); if (m == 0) return a; return d3(a.x / m, a.y / m, a.z / m); }
__device__ __forceinline__ D3 sub3(D3 a, D3 b) { return d3(a.x - b.x, a.y - b.y, a.z - b.z); }
__device__ __forceinline__ D3 add3(D3 a, D3 b) { return d3(a.x + b.x, a.y + b.y, a.z + b.z); }
__device__ __forceinline__ D3 scale3(D3 a, double s) { return d3(a.x * s, a.y * s, a.z * s); }
// myMatrix.multVert with w = 1 / w = 0 (the leading "0 +" and trailing "* 1" of the reference loop are exact)
__device__ __forceinline__ D3 xfPoint(const double* __restrict__ m, D3 p) {
  return d3((((m[0] * p.x) + (m[1] * p.y)) + (m[2] * p.z)) + m[3], (((m[4] * p.x) + (m[5] * p.y)) + (m[6] * p.z)) + m[7], (((m[8] * p.x) + (m[9] * p.y)) + (m[10] * p.z)) + m[11]);
}
__device__ __forceinline__ D3 xfVector(const double* __restrict__ m, D3 p) {
  return d3(((m[0] * p.x) + (m[1] * p.y)) + (m[2] * p.z), ((m[4] * p.x) + (m[5] * p.y)) + (m[6] * p.z), ((m[8] * p.x) + (m[9] * p.y)) + (m[10] * p.z));
}
__device__ __forceinline__ double jminD(double a, double b) { if (a != a) return a; if (b != b) return b; return a < b ? a : b; }
__device__ __forceinline__ double jmaxD(double a, double b) { if (a != a) return a; if (b != b) return b; return a > b ? a : b; }
__device__ __forceinline__ int j2iD(double d) { if (d != d) return 0; if (d >= 2147483647.0) return 2147483647; if (d <= -2147483648.0) return (int)0x80000000; return (int)d; }
__device__ __forceinline__ int fastfloorD(double x) { return x > 0 ? j2iD(x) : j2iD(x) - 1; }
__device__ __forceinline__ int fastfloorF(float x) { return x > 0 ? j2iD((double)x) : j2iD((double)x) - 1; }

// DistRayTracer.rotVecAroundAxis (:336-349)
__device__ inline D3 rotAboutAxis(D3 v, D3 u, double th) {
  double c = cos(th), s = sin(th), omc = 1 - c;
  double ux2 = u.x * u.x, uy2 = u.y * u.y, uz2 = u.z * u.z, uxy = u.x * u.y, uxz = u.x * u.z, uyz = u.y * u.z;
  double uzS = u.z * s, uyS = u.y * s, uxS = u.x * s, uxzC = uxz * omc, uxyC = uxy * omc, uyzC = uyz * omc;
  return d3((ux2 * omc + c) * v.x + (uxyC - uzS) * v.y + (uxzC + uyS) * v.z,
            (uxyC + uzS) * v.x + (uy2 * omc + c) * v.y + (uyzC - uxS) * v.z,
            (uxzC - uyS) * v.x + (uyzC + uxS) * v.y + (uz2 * omc + c) * v.z);
}

// ---- Philox4x32-10 keyed sampler; same function as the oracle's (tests assert bit equality through drt_sample_u01)
enum : uint32_t { STREAM_PIXEL = 0x0u, STREAM_PHOTON = 0x50484F54u };
enum : uint32_t { DIM_AA_Y = 0, DIM_AA_X = 1, DIM_TIME = 2, DIM_LENS_ANGLE = 3, DIM_LENS_RADIUS = 4, DIM_LIGHT_BASE = 16, DIM_LIGHT_STRIDE = 8 };
__host__ __device__ inline double philoxU01(uint64_t seed, uint32_t stream, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  uint32_t c0 = a, c1 = b, c2 = c, c3 = d, k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32) ^ stream;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
    uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0, n1 = (uint32_t)p1, n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1, n3 = (uint32_t)p0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3; k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  uint64_t hi = c0 >> 5, lo = c1 >> 6;
  return (double)((hi << 26) | lo) * (1.0 / 9007199254740992.0);
}
// ThreadLocalRandom.nextDouble(origin, bound)
__device__ __forceinline__ double urange(double u, double origin, double bound) {
  double r = u * (bound - origin) + origin;
  if (r >= bound) r = __longlong_as_double(__double_as_longlong(bound) + (bound > 0 ? -1 : 1));   // Math.nextDown for the bounds used here (never 0)
  return r;
}

// device view of the flattened scene (all pointers into HBM)
struct DScene {
  const FXform* xforms; const FPrim* prims; const double* pdata; const FObjRef* top; const FObjRef* children;
  const FInstance* instances; const FList* lists; const FBvh* bvhs; const FNode* nodes; const FLight* lights;
  const double* lightPos;           // xfPoint(CTM, origin) of every light, 3 doubles each: formed on the device once per upload (k_light_pos)
  const FShader* shaders; const FTexture* textures; const double* texColors; const FImage* images; const int32_t* texels;
  // fast-BVH view: packed triangles and the node array their fastRoot indexes (== nodes, or the GPU-built LBVH nodes); accelMode = drt.h DRT_ACCEL_*
  const FTri* tris; const FNode* fnodes; const FNode32* fnodes32; int32_t accelMode; int32_t padA;
  // photon map (hash grid), see photon kernels
  const double* phPos; const double* phPwr; const uint32_t* cellStart; const float* phPos32; uint32_t gridDim[3]; uint32_t numPhotons; double gridMin[3]; double cellSize;
  float phAbsMax; float padP;      // phPos32: float4 mirror of phPos (pre-test of the gather); phAbsMax: largest |coordinate| of a stored photon, rounded up
  FGlobals g;
};

}  // namespace drt
