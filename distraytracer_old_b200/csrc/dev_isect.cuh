// Ray / primitive intersection and the reference-exact ("literal") traversal.
//
// Replaces (reference file:line, /root/reference/src/rayTracerDistAccelShdPhtnMap/):
//   myRay.java:91-102            getTransformedRay (in-place normalisation of the source ray, SURVEY Q7)
//   myGeomBase.java:132-162      myBBox.intersectCheck, "entry t > 0" rule (SURVEY Q1)
//   myPlanarObject.java:104-115,165-211  plane hit + inside test, stateless two-sidedness (SURVEY Q9)
//   myImpObject.java:76-94,174-192,259-302  sphere / open cylinder / capped cylinder
//   myScene.java:879-903         calcShadow / findClosestRayHit over the top-level list
//   myGeomBase.java:216-222,268-302,397-421  root gate, list loops, ordered BVH recursion (SURVEY Q4)
//   mySceneObject.java:33-38,117-127  shadow rule, instance forwarding (SURVEY Q7,Q8)
#pragma once
#include "dev_math.cuh"

namespace drt {

// origin, "direction" vector (may be re-normalised in place), "dirAra" copy (never re-normalised) -- myRay.java:14-18
struct Ray { D3 o, d, a; bool norm; };

struct alignas(16) Hit {
  double t;
  int32_t prim, arg0, arg1, state;        // state: polygon winding state used (0/1[/2 for planes])
  int32_t hitXform, shaderOverride, inst, pad0;
  D3 loc;                                  // hit point in the primitive's space (rayHit.hitLoc)
  D3 rawDir;                               // rayHit.fwdTransRayDir (SURVEY Q8)
  double pad1;
};
// what a primitive test reports; the caller fills the Hit record only for candidates that win
struct PHit { double t; int32_t arg0, arg1, state, boxRaw; };
// pad0 during a closest-hit search: 2 (list child index + 1) + boxRaw, where the winner came from (closestHitT forms loc / rawDir from it)
__device__ __forceinline__ void takeHit(const DScene& S, Hit& dst, const PHit& ph, int primIdx, const Ray& r, D3 rawDir, int hitXform) {
  dst.t = ph.t; dst.prim = primIdx; dst.arg0 = ph.arg0; dst.arg1 = ph.arg1; dst.state = ph.state; dst.hitXform = hitXform; dst.shaderOverride = -1; dst.inst = -1;
  dst.pad0 = ph.boxRaw ? 1 : 0;
  dst.loc = d3((r.d.x * ph.t) + r.o.x, (r.d.y * ph.t) + r.o.y, (r.d.z * ph.t) + r.o.z);       // transRay.pointOnRay(t), myRay.java:82-87
  // rendered box: the direction recorded in the hit is CTM x transformed direction (myGeomBase.java:160)
  dst.rawDir = ph.boxRaw ? xfVector(S.xforms[S.prims[primIdx].xform].m, r.d) : rawDir;
}
__device__ __forceinline__ void hitReset(Hit& h) { h.t = DRT_DMAX; h.prim = -1; h.arg0 = 0; h.arg1 = 0; h.state = 0; h.hitXform = -1; h.shaderOverride = -1; h.inst = -1; h.pad0 = 0; h.loc = d3(0, 0, 0); h.rawDir = d3(0, 0, 0); h.pad1 = 0; }

struct TraceCounters { unsigned long long box, prim; };

// device-side error word, reset and checked by the host around every render / probe / photon call:
//   DEV_ERR_INCOMPLETE  a search ran beyond its capacity (traversal stack, photon candidate ranges): the result would silently miss
//                       something, so the call fails instead
//   DEV_ERR_QUEUE       a bounce level overflowed its queue or the node pool: the host renders the frame again with smaller batches
//   DEV_ERR_DEPTH       rays reached a level the call did not launch: the host renders the frame again with full depth
constexpr unsigned int DEV_ERR_INCOMPLETE = 1u, DEV_ERR_QUEUE = 2u, DEV_ERR_DEPTH = 4u;
__device__ unsigned int g_devError;
__device__ __forceinline__ void flagError(unsigned int bit) { if (!(g_devError & bit)) atomicOr(&g_devError, bit); }

__device__ __forceinline__ Ray makeRay(D3 o, D3 dirNormalized) { Ray r; r.o = o; r.d = dirNormalized; r.a = dirNormalized; r.norm = true; return r; }
// getTransformedRay: normalise the source direction in place (only if it is not already unit length: canonical mode,
// see DESIGN.md "re-normalisation"), transform origin as a point and direction as a vector, do NOT normalise the result.
__device__ __forceinline__ Ray xfRay(Ray& src, const double* __restrict__ inv) {
  if (!src.norm) { src.d = norm3(src.d); src.norm = true; }
  Ray r; r.o = xfPoint(inv, src.o); r.d = xfVector(inv, src.d); r.a = r.d; r.norm = false; return r;
}
__device__ __forceinline__ D3 pointOnRay(const Ray& r, double t) { return d3((r.d.x * t) + r.o.x, (r.d.y * t) + r.o.y, (r.d.z * t) + r.o.z); }

// ---- slab test, literal (true divisions, running min/max that NaN never replaces)
__device__ __forceinline__ bool boxTest(const double* __restrict__ mn, const double* __restrict__ mx, const Ray& r, double& tEntry, int& face) {
  double o[3] = {r.o.x, r.o.y, r.o.z}, d[3] = {r.a.x, r.a.y, r.a.z};
  double tMin[3], tMax[3], biggestMin = -DRT_DMAX; int idx = -1;
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    double v1 = (mn[i] - o[i]) / d[i], v2 = (mx[i] - o[i]) / d[i];
    if (v1 < v2) { tMin[i] = v1; tMax[i] = v2; if (biggestMin < v1) { idx = i; biggestMin = v1; } }
    else { tMin[i] = v2; tMax[i] = v1; if (biggestMin < v2) { idx = i + 3; biggestMin = v2; } }
  }
  double minMax = DRT_DMAX, maxMin = -DRT_DMAX;
#pragma unroll
  for (int i = 0; i < 3; ++i) { if (tMax[i] < minMax) minMax = tMax[i]; if (tMin[i] > maxMin) maxMin = tMin[i]; }
  if ((minMax > maxMin) && biggestMin > 0) { tEntry = biggestMin; face = idx; return true; }
  return false;
}

// Same decisions and the same entry t as boxTest(), bit for bit, at a fraction of the FP64 divisions:
// the six slab values are first formed with a per-ray reciprocal (<= 2 ulp from the quotient the reference computes);
// every comparison the reference makes (v1<v2 per axis, min(tMax) > max(tMin), entry > 0, which tMin is largest) is accepted
// only when the operands are separated by far more than that error; the one value that leaves the function (entry t) is then
// recomputed with the reference's own division.  Anything closer than the margin falls back to the literal test.
#define DRT_CLEAR(a, b) (fabs((a) - (b)) > 1e-14 * (fabs(a) + fabs(b)))
__device__ __forceinline__ bool boxTestFx(const double* __restrict__ mn, const double* __restrict__ mx, const Ray& r, const D3& inv, double& tEntry) {
  const double nx1 = mn[0] - r.o.x, nx2 = mx[0] - r.o.x, ny1 = mn[1] - r.o.y, ny2 = mx[1] - r.o.y, nz1 = mn[2] - r.o.z, nz2 = mx[2] - r.o.z;
  const double ax1 = nx1 * inv.x, ax2 = nx2 * inv.x, ay1 = ny1 * inv.y, ay2 = ny2 * inv.y, az1 = nz1 * inv.z, az2 = nz2 * inv.z;
  const bool sx = ax1 < ax2, sy = ay1 < ay2, sz = az1 < az2;
  const double tnx = sx ? ax1 : ax2, tfx = sx ? ax2 : ax1, tny = sy ? ay1 : ay2, tfy = sy ? ay2 : ay1, tnz = sz ? az1 : az2, tfz = sz ? az2 : az1;
  double far_ = tfx; if (tfy < far_) far_ = tfy; if (tfz < far_) far_ = tfz;
  double near_ = tnx; int ax = 0; if (tny > near_) { near_ = tny; ax = 1; } if (tnz > near_) { near_ = tnz; ax = 2; }
  const double second = (ax == 0) ? (tny > tnz ? tny : tnz) : (ax == 1 ? (tnx > tnz ? tnx : tnz) : (tnx > tny ? tnx : tny));
  // all operands finite and every decision clear of the reciprocal's error?
  const bool ok = DRT_CLEAR(ax1, ax2) && DRT_CLEAR(ay1, ay2) && DRT_CLEAR(az1, az2) && DRT_CLEAR(far_, near_) && DRT_CLEAR(near_, second) && (fabs(near_) > 1e-290) && (fabs(far_) < 1e290) && (fabs(near_) < 1e290);
  if (!ok) { int face; return boxTest(mn, mx, r, tEntry, face); }
  if (!((far_ > near_) && near_ > 0)) return false;
  // entry t exactly as the reference forms it: (bound - origin) / direction on the winning axis
  const double num = (ax == 0) ? (sx ? nx1 : nx2) : (ax == 1 ? (sy ? ny1 : ny2) : (sz ? nz1 : nz2));
  const double den = (ax == 0) ? r.a.x : (ax == 1 ? r.a.y : r.a.z);
  tEntry = num / den;
  return true;
}
__device__ __forceinline__ D3 rayInv(const Ray& r) { return d3(1.0 / r.a.x, 1.0 / r.a.y, 1.0 / r.a.z); }

// Division-free accept/reject of the same rule.  The six slab values formed with the per-ray reciprocal are within 1.5 * 2^-52 (relative)
// of the quotients the reference forms; min/max selection is 1-Lipschitz, so near_/far_ carry the same bound relative to their own size.
// Returns 1 (accepted: min(tMax) > max(tMin) and entry > 0, beyond doubt), 0 (rejected beyond doubt) or -1 (inside the error margin, or
// NaN/inf/denormal operands: the caller runs the exact test).  nearApprox is the entry t to ~3e-16 relative -- good enough to ORDER and
// PRUNE conservatively, never used where the reference's own value decides something.
__device__ __forceinline__ int boxQuick(const double* __restrict__ mn, const double* __restrict__ mx, const Ray& r, const D3& inv, double& nearApprox) {
  const double ax1 = (mn[0] - r.o.x) * inv.x, ax2 = (mx[0] - r.o.x) * inv.x, ay1 = (mn[1] - r.o.y) * inv.y, ay2 = (mx[1] - r.o.y) * inv.y, az1 = (mn[2] - r.o.z) * inv.z, az2 = (mx[2] - r.o.z) * inv.z;
  const bool sx = ax1 < ax2, sy = ay1 < ay2, sz = az1 < az2;
  const double tnx = sx ? ax1 : ax2, tfx = sx ? ax2 : ax1, tny = sy ? ay1 : ay2, tfy = sy ? ay2 : ay1, tnz = sz ? az1 : az2, tfz = sz ? az2 : az1;
  double far_ = tfx; if (tfy < far_) far_ = tfy; if (tfz < far_) far_ = tfz;
  double near_ = tnx; if (tny > near_) near_ = tny; if (tnz > near_) near_ = tnz;
  nearApprox = near_;                       // defined on every return path (callers scale it before looking at the verdict)
  if (!(fabs(near_) > 1e-290) || !(fabs(far_) < 1e290) || !(fabs(near_) < 1e290)) return -1;
  const double tol = 1e-14 * (fabs(far_) + fabs(near_)), gap = far_ - near_;
  if (gap > tol) return near_ > 0 ? 1 : 0;
  return (-gap > tol) ? 0 : -1;
}
// box accepted AND (dist - entry) > eps, the shadow-ray form (myGeomBase.java:166-170,268-269,397-404)
__device__ __forceinline__ bool boxAcceptShadow(const double* __restrict__ mn, const double* __restrict__ mx, const Ray& r, const D3& inv, double dist) {
  double te; const int q = boxQuick(mn, mx, r, inv, te);
  if (q == 0) return false;
  if (q > 0) { const double diff = dist - te, m = 1e-13 * (fabs(dist) + fabs(te)); if (diff > DRT_EPS + m) return true; if (diff < DRT_EPS - m) return false; }
  return boxTestFx(mn, mx, r, inv, te) && (dist - te) > DRT_EPS;
}

// accepted?  (the entry t is not needed: root gates, left children of the literal recursion)
__device__ __forceinline__ bool boxHit(const double* __restrict__ mn, const double* __restrict__ mx, const Ray& r, const D3& inv) {
  double te; const int q = boxQuick(mn, mx, r, inv, te);
  if (q >= 0) return q != 0;
  int face; return boxTest(mn, mx, r, te, face);
}
// accepted AND (no hit yet OR entry t < tCur): the right-child rule of myBVH.traverseStruct (myGeomBase.java:413-417); the exact entry t is
// formed only when the approximate one is within 1e-13 (relative) of tCur
__device__ __forceinline__ bool boxHitBefore(const double* __restrict__ mn, const double* __restrict__ mx, const Ray& r, const D3& inv, double tCur) {
  double te; const int q = boxQuick(mn, mx, r, inv, te);
  if (q == 0) return false;
  if (q > 0) { if (!(tCur < DRT_DMAX)) return true; const double m = 1e-13 * (fabs(te) + fabs(tCur)); if (te < tCur - m) return true; if (te > tCur + m) return false; }
  if (!boxTestFx(mn, mx, r, inv, te)) return false;
  return !(tCur < DRT_DMAX) || te < tCur;
}

// ---- primitives. `r` is the ray in the primitive's space, rawDir the direction recorded in the hit.
// Returns true and fills h (t, loc, args, state) on a hit. time: ray time for moving spheres.
__device__ __noinline__ bool primTest(const DScene& S, int primIdx, const Ray& r, double time, PHit& h) {
  h.boxRaw = 0;
  const FPrim P = S.prims[primIdx];
  const double* __restrict__ q = S.pdata + P.data;
  switch (P.type) {
    case PT_SPHERE: case PT_MOVSPHERE: {
      D3 c = d3(q[0], q[1], q[2]); double rx = q[3], ry = q[4], rz = q[5];
      if (P.type == PT_MOVSPHERE) { D3 bMa = d3(q[6] - c.x, q[7] - c.y, q[8] - c.z); c = d3(c.x + time * bMa.x, c.y + time * bMa.y, c.z + time * bMa.z); }
      double dxr = r.d.x / rx, dyr = r.d.y / ry, dzr = r.d.z / rz;
      double a = ((dxr) * (dxr)) + ((dyr) * (dyr)) + ((dzr) * (dzr));
      D3 pC = d3((r.o.x - c.x) / rx, (r.o.y - c.y) / ry, (r.o.z - c.z) / rz);
      double b = 2 * (((dxr) * pC.x) + ((dyr) * pC.y) + ((dzr) * pC.z));
      double cc = (pC.x * pC.x) + (pC.y * pC.y) + (pC.z * pC.z) - 1;
      double ta = 2 * a, discr = ((b * b) - (2 * ta * cc));
      if (!(discr < 0)) {
        double d1 = sqrt(discr), t1 = (-1 * b + d1) / (ta), t2 = (-1 * b - d1) / (ta);
        double tv = jminD(t1, t2);
        if (tv < DRT_EPS) { tv = jmaxD(t1, t2); if (tv < DRT_EPS) return false; }
        h.t = tv; h.arg0 = 0; h.arg1 = 0; h.state = 0; return true;
      }
      return false;
    }
    case PT_TRI: case PT_QUAD: {
      const int n = (P.type == PT_TRI) ? 3 : 4, stride = (P.type == PT_TRI) ? DRT_TRI_STATE : DRT_QUAD_STATE;
      int st = 0; const double* __restrict__ s = q;
      D3 N = d3(s[3 * n], s[3 * n + 1], s[3 * n + 2]);
      double planeRes = dot3(N, r.d);
      if (!(fabs(planeRes) > 0)) return false;
      if (planeRes > 0) {                       // invertNormal(): continue with the reversed winding
        st = 1; s = q + stride; N = d3(s[3 * n], s[3 * n + 1], s[3 * n + 2]); planeRes = dot3(N, r.d);
        if (!(fabs(planeRes) > 0) || planeRes > 0) return false;
      }
      double t = -(dot3(N, r.o) + s[3 * n + 3]) / planeRes;
      if (!(t > DRT_EPS)) return false;
      D3 p = pointOnRay(r, t);
#pragma unroll 1
      for (int i = 0; i < n; ++i) {
        int pi = (i == 0 ? n - 1 : i - 1);
        D3 vi = d3(s[3 * i], s[3 * i + 1], s[3 * i + 2]), vp = d3(s[3 * pi], s[3 * pi + 1], s[3 * pi + 2]);
        D3 ir = d3(p.x - vi.x, p.y - vi.y, p.z - vi.z), e = d3(vi.x - vp.x, vi.y - vp.y, vi.z - vp.z);
        D3 tmp = cross3(ir, e);
        if (dot3(tmp, N) < -DRT_EPS) return false;
      }
      h.t = t; h.arg0 = 0; h.arg1 = 0; h.state = st; return true;
    }
    case PT_PLANE: {
      int st = 0; D3 N = d3(q[0], q[1], q[2]); double D = q[3];
      double planeRes = dot3(N, r.d);
      if (!(fabs(planeRes) > 0)) return false;
      if (planeRes > 0) { st = 1; N = d3(q[4], q[5], q[6]); D = q[7]; planeRes = dot3(N, r.d); if (!(fabs(planeRes) > 0)) return false;
        if (planeRes > 0) { st = 2; N = d3(q[8], q[9], q[10]); D = q[11]; planeRes = dot3(N, r.d); if (!(fabs(planeRes) > 0) || planeRes > 0) return false; } }
      double t = -(dot3(N, r.o) + D) / planeRes;
      if (!(t > DRT_EPS)) return false;
      h.t = t; h.arg0 = 0; h.arg1 = 0; h.state = st; return true;
    }
    case PT_HCYL: {
      double cx = q[0], cz = q[2], radX = q[3], radZ = q[4], yTop = q[5], yBot = q[6];
      double dxr = r.d.x / radX, dzr = r.d.z / radZ, pcx = (r.o.x - cx) / radX, pcz = (r.o.z - cz) / radZ;
      double a = ((dxr) * (dxr)) + ((dzr) * (dzr)), b = 2 * (((dxr) * pcx) + ((dzr) * pcz)), c = (pcx * pcx) + (pcz * pcz) - 1;
      double discr = ((b * b) - (4 * a * c));
      if (!(discr < 0)) {
        double d1 = sqrt(discr), t1 = (-b + d1) / (2 * a), t2 = (-b - d1) / (2 * a);
        double tv = jminD(t1, t2), to = jmaxD(t1, t2);
        if (tv < -DRT_EPS) { double tmp = to; to = tv; tv = tmp; if (tv < -DRT_EPS) return false; }
        double y1 = r.o.y + (tv * r.d.y);
        if ((tv > DRT_EPS) && (y1 > yBot) && (y1 < yTop)) { h.t = tv; h.arg0 = 0; h.arg1 = 0; h.state = 0; return true; }
        double y2 = r.o.y + (to * r.d.y);
        if ((to > DRT_EPS) && (y2 > yBot) && (y2 < yTop)) { h.t = to; h.arg0 = 1; h.arg1 = 0; h.state = 0; return true; }
      }
      return false;
    }
    case PT_CYL: {
      double cx = q[0], cz = q[2], radX = q[3], radZ = q[4], yTop = q[5], yBot = q[6];
      double dxr = r.d.x / radX, dzr = r.d.z / radZ, pcx = (r.o.x - cx) / radX, pcz = (r.o.z - cz) / radZ;
      double a = ((dxr) * (dxr)) + ((dzr) * (dzr)), b = 2 * (((dxr) * pcx) + ((dzr) * pcz)), c = (pcx * pcx) + (pcz * pcz) - 1;
      double discr = ((b * b) - (4 * a * c));
      if (!(discr < 0)) {
        double d1 = sqrt(discr), t1 = (-b + d1) / (2 * a), t2 = (-b - d1) / (2 * a);
        double cv = jminD(t1, t2), co = jmaxD(t1, t2);
        if (cv < DRT_EPS) { co = cv; cv = jmaxD(t1, t2); if (cv < DRT_EPS) return false; }
        bool planeRes = true; double pl[2];
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          const double* e = q + 7 + 4 * i;
          double den = e[0] * r.d.x + e[1] * r.d.y + e[2] * r.d.z;
          if (fabs(den) > DRT_EPS) { double num = e[0] * r.o.x + e[1] * r.o.y + e[2] * r.o.z + e[3]; pl[i] = -num / den; } else pl[i] = 10000;
        }
        double pv = jminD(pl[0], pl[1]); int vis = (pv == pl[0] ? 0 : 1);
        if (pv < 0) { pv = pl[vis]; if (pv < DRT_EPS) planeRes = false; }
        double tv, mxC = jmaxD(cv, co), mnC = jminD(cv, co);
        if (planeRes && (((mnC <= 0) && (pv >= -DRT_EPS) && (pv <= mxC)) || ((pv > mnC) && (pv <= mxC)))) tv = pv; else { tv = cv; vis = 2; }
        double y1 = r.o.y + (tv * r.d.y);
        if ((y1 + DRT_EPS >= yBot) && (y1 - DRT_EPS <= yTop)) { h.t = tv; h.arg0 = vis; h.arg1 = 0; h.state = 0; return true; }
      }
      return false;
    }
    case PT_BOX: {
      double t; int face; if (!boxTest(q, q + 3, r, t, face)) return false;
      h.t = t; h.arg0 = 0; h.arg1 = face; h.state = 0; h.boxRaw = 1; return true;
    }
    // ---- extension primitives (no reference arithmetic to follow: the semantics are defined here; the test suite holds a CPU twin, DESIGN.md section 8)
    case PT_QUADRIC: {
      const double a = q[0], b = q[1], c = q[2], d = q[3], e = q[4], f = q[5], g = q[6], hh = q[7], ii = q[8], j = q[9];
      const double ox = r.o.x, oy = r.o.y, oz = r.o.z, dx = r.d.x, dy = r.d.y, dz = r.d.z;
      const double A = (((((a * dx) * dx) + ((b * dy) * dy)) + ((c * dz) * dz)) + ((d * dx) * dy)) + (((e * dx) * dz) + ((f * dy) * dz));
      const double B = ((2 * ((((a * ox) * dx) + ((b * oy) * dy)) + ((c * oz) * dz))) + (((d * ((ox * dy) + (oy * dx))) + (e * ((ox * dz) + (oz * dx)))) + (f * ((oy * dz) + (oz * dy))))) + (((g * dx) + (hh * dy)) + (ii * dz));
      const double C = ((((((a * ox) * ox) + ((b * oy) * oy)) + ((c * oz) * oz)) + ((d * ox) * oy)) + (((e * ox) * oz) + ((f * oy) * oz))) + ((((g * ox) + (hh * oy)) + (ii * oz)) + j);
      double t0, t1; int nr;
      if (A == 0) { if (B == 0) return false; t0 = -C / B; t1 = t0; nr = 1; }
      else {
        const double disc = (B * B) - ((4 * A) * C); if (disc < 0) return false;
        const double sq = sqrt(disc), ta = (-B - sq) / (2 * A), tb = (-B + sq) / (2 * A); t0 = jminD(ta, tb); t1 = jmaxD(ta, tb); nr = 2;
      }
      for (int k = 0; k < nr; ++k) {
        const double t = k == 0 ? t0 : t1; if (!(t > DRT_EPS)) continue;
        const double px = (dx * t) + ox, py = (dy * t) + oy, pz = (dz * t) + oz;
        if (px < q[10] || py < q[11] || pz < q[12] || px > q[13] || py > q[14] || pz > q[15]) continue;
        h.t = t; h.arg0 = k; h.arg1 = 0; h.state = 0; return true;
      }
      return false;
    }
    case PT_TORUS: {
      // (|p|^2 + R^2 - r^2)^2 = 4 R^2 (px^2 + pz^2), p = o + t d relative to the centre: quartic c4 t^4 + ... + c0.  Smallest root > eps, found
      // inside the ray's span of the bounding sphere |p| <= 1.001 (R + r) by a fixed scan (64 steps) for the first sign change + 64 bisection steps.
      const double R = q[3], rr = q[4];
      const double ox = r.o.x - q[0], oy = r.o.y - q[1], oz = r.o.z - q[2], dx = r.d.x, dy = r.d.y, dz = r.d.z;
      const double al = ((dx * dx) + (dy * dy)) + (dz * dz), be = ((ox * dx) + (oy * dy)) + (oz * dz), oo = ((ox * ox) + (oy * oy)) + (oz * oz);
      if (!(al > 0)) return false;
      const double Rb = (R + rr) * 1.001, dsc = (be * be) - (al * (oo - (Rb * Rb))); if (dsc < 0) return false;
      const double sq = sqrt(dsc); double ta = (-be - sq) / al, tb = (-be + sq) / al;
      if (!(tb > DRT_EPS)) return false; if (ta < DRT_EPS) ta = DRT_EPS;
      const double kk = oo + ((R * R) - (rr * rr)), R4 = 4 * (R * R);
      const double c4 = al * al, c3 = 4 * (al * be), c2 = ((2 * (al * kk)) + (4 * (be * be))) - (R4 * ((dx * dx) + (dz * dz))), c1 = (4 * (be * kk)) - ((2 * R4) * ((ox * dx) + (oz * dz))), c0 = (kk * kk) - (R4 * ((ox * ox) + (oz * oz)));
      auto F = [&](double t) { return ((((((c4 * t) + c3) * t) + c2) * t + c1) * t) + c0; };
      const double step = (tb - ta) / 64; double lo = ta, flo = F(lo); bool found = false; double hi = ta;
      for (int k = 1; k <= 64; ++k) { hi = (k == 64) ? tb : ta + (step * k); const double fhi = F(hi); if ((flo > 0) != (fhi > 0)) { found = true; break; } lo = hi; flo = fhi; }
      if (!found) return false;
      for (int k = 0; k < 64; ++k) { const double mid = 0.5 * (lo + hi), fm = F(mid); if ((fm > 0) == (flo > 0)) { lo = mid; flo = fm; } else hi = mid; }
      const double t = 0.5 * (lo + hi); if (!(t > DRT_EPS)) return false;
      h.t = t; h.arg0 = 0; h.arg1 = 0; h.state = 0; return true;
    }
  }
  return false;
}

// ---------------------------------------------------------------------------------------------------------------
// fast BVHs: packed triangles, both child boxes per node, near-first ordered descent with global pruning
// ---------------------------------------------------------------------------------------------------------------
// conventional conservative slab test (LBVH mode only): a ray that starts inside the box enters it at t = 0.  fmin / fmax pick the near and
// far plane of each axis whatever the sign of the direction, and drop the NaN slab value of an axis-parallel ray whose origin lies on a plane
__device__ __forceinline__ bool boxTestStd(const double* mn, const double* mx, const Ray& r, const D3& inv, double& tEntry) {
  double t0 = (mn[0] - r.o.x) * inv.x, t1 = (mx[0] - r.o.x) * inv.x; double tn = fmin(t0, t1), tf = fmax(t0, t1);
  t0 = (mn[1] - r.o.y) * inv.y; t1 = (mx[1] - r.o.y) * inv.y; tn = fmax(tn, fmin(t0, t1)); tf = fmin(tf, fmax(t0, t1));
  t0 = (mn[2] - r.o.z) * inv.z; t1 = (mx[2] - r.o.z) * inv.z; tn = fmax(tn, fmin(t0, t1)); tf = fmin(tf, fmax(t0, t1));
  tEntry = fmax(tn, 0.0); return tf >= tEntry;
}

// The traversal bodies are force-inlined in the lean kernels so that ray and hit records stay in registers; -DDRT_LEAN_INLINE=__noinline__ builds the
// outlined form, which passes the same equivalence tests (DESIGN.md section 3, `__noinline__` note).
#ifndef DRT_LEAN_INLINE
#define DRT_LEAN_INLINE __forceinline__
#endif
#define DRT_FSTACK 64            // traversal stack of the generic kernels
// Compile-time feature set of a tracing kernel (see render.cu): the lean kernels carry only the code their scene shape needs -- a small
// local frame and register budget -- and hand the rare ray they cannot serve (axis-parallel direction, mixed units through an instance,
// traversal deeper than the short stack) to the generic kernel through a deferral list.  Every ray is traced start to finish by ONE variant,
// and all variants implement the same rules, so results do not depend on which one served a ray.
enum : int { TF_LITERAL1 = 1,     // literal (reference-order) BVH recursion at the top level, lists holding instanced accels
             TF_LEVEL2 = 2,       // literal recursion inside instanced accels
             TF_ALL = 7 };        // the generic variant: serves every ray, whatever its direction
#ifndef DRT_LSTACK
#define DRT_LSTACK 32            // short traversal stack of the lean kernels (a <=5-per-leaf median tree over 2^24 triangles is 23 deep)
#endif
__device__ __forceinline__ int32_t childRef(int32_t link, int32_t triCode) { return link >= 0 ? link : ~triCode; }

// exact (true-division) box test, out of line; returns the entry t (> 0 by the acceptance rule) or -1 when the box is rejected.  The value
// travels in the return register: a `double&` result would force the callers' entry-t variables into local memory on EVERY node visit.
__device__ __noinline__ double boxExactEntry(const double* __restrict__ box6, double ox, double oy, double oz, double ax, double ay, double az) {
  Ray r; r.o = d3(ox, oy, oz); r.a = d3(ax, ay, az); r.d = r.a; r.norm = false; int face; double te;
  double b[6]; for (int i = 0; i < 6; ++i) b[i] = __ldg(box6 + i);
  return boxTest(b, b + 3, r, te, face) ? te : -1.0;
}
// conventional slab test (LBVH mode) out of line: entry t (>= 0) or -1.  ANY_DIR (generic kernels): boxTestStd's fmin / fmax, right for every
// direction.  Otherwise (lean kernels, regular directions only) the near and far plane of each axis are picked by the sign of the direction: the
// same slab values and decisions.  The lean form is kept because the fmin / fmax body changes the lean kernels' register allocation, which
// measured 1.9 % slower per frame on plnts3ColsBunnies 4K (B200).
template <bool ANY_DIR>
__device__ __noinline__ double boxStdEntry(const double* __restrict__ box6, double ox, double oy, double oz, double ax, double ay, double az) {
  if constexpr (ANY_DIR) {
    Ray r; r.o = d3(ox, oy, oz); r.a = d3(ax, ay, az); r.d = r.a; r.norm = false; double te;
    double b[6]; for (int i = 0; i < 6; ++i) b[i] = __ldg(box6 + i);
    return boxTestStd(b, b + 3, r, rayInv(r), te) ? te : -1.0;
  } else {
    const double ix = 1.0 / ax, iy = 1.0 / ay, iz = 1.0 / az; const bool px = ax > 0, py = ay > 0, pz = az > 0;
    const double mnx = __ldg(box6), mny = __ldg(box6 + 1), mnz = __ldg(box6 + 2), mxx = __ldg(box6 + 3), mxy = __ldg(box6 + 4), mxz = __ldg(box6 + 5);
    const double nx = ((px ? mnx : mxx) - ox) * ix, fx = ((px ? mxx : mnx) - ox) * ix;
    const double ny = ((py ? mny : mxy) - oy) * iy, fy = ((py ? mxy : mny) - oy) * iy;
    const double nz = ((pz ? mnz : mxz) - oz) * iz, fz = ((pz ? mxz : mnz) - oz) * iz;
    double near_ = nx > ny ? nx : ny; near_ = nz > near_ ? nz : near_; near_ = near_ > 0.0 ? near_ : 0.0;
    double far_ = fx < fy ? fx : fy; far_ = fz < far_ ? fz : far_;
    return far_ >= near_ ? near_ : -1.0;
  }
}
// directions the lean kernels serve: every component finite, non-zero and of sane magnitude (all but axis-parallel rays)
__device__ __forceinline__ bool regularDir(D3 a) {
  const double x = fabs(a.x), y = fabs(a.y), z = fabs(a.z);
  return x > 1e-100 && x < 1e100 && y > 1e-100 && y < 1e100 && z > 1e-100 && z < 1e100;
}
// myTriangle.intersectCheck on a packed record: the same operations, in the same order, as primTest's PT_TRI case, with one shortcut that
// cannot change the outcome: a plane hit farther than the best hit so far is dropped before the inside test (the reference would compute it
// and then discard it in `t < closest`)
__device__ __forceinline__ bool leanTri(const FTri* __restrict__ T, double ox, double oy, double oz, double dx, double dy, double dz, double bestT, double& tOut, int& stOut, int32_t& rank) {
  const double2* __restrict__ q = reinterpret_cast<const double2*>(T);
  const double2 q4 = __ldg(q + 4), q5 = __ldg(q + 5), q6 = __ldg(q + 6);                    // (v8, N.x) (N.y, N.z) (D, Drev)
  double Nx = q4.y, Ny = q5.x, Nz = q5.y, D = q6.x;
  double planeRes = ((Nx * dx) + (Ny * dy)) + (Nz * dz);
  if (!(fabs(planeRes) > 0)) return false;
  int st = 0;
  if (planeRes > 0) { st = 1; Nx = -Nx; Ny = -Ny; Nz = -Nz; D = q6.y; planeRes = -planeRes; }
  const double t = -((((Nx * ox) + (Ny * oy)) + (Nz * oz)) + D) / planeRes;
  if (!(t > DRT_EPS) || t > bestT) return false;
  const double2 q0 = __ldg(q), q1 = __ldg(q + 1), q2 = __ldg(q + 2), q3 = __ldg(q + 3);     // (v0 v1) (v2 v3) (v4 v5) (v6 v7)
  const double px = (dx * t) + ox, py = (dy * t) + oy, pz = (dz * t) + oz;
  const double ax_ = q0.x, ay_ = q0.y, az_ = q1.x, bx_ = q1.y, by_ = q2.x, bz_ = q2.y, cx_ = q3.x, cy_ = q3.y, cz_ = q4.x;
  const double V0x = st ? cx_ : ax_, V0y = st ? cy_ : ay_, V0z = st ? cz_ : az_, V2x = st ? ax_ : cx_, V2y = st ? ay_ : cy_, V2z = st ? az_ : cz_;
  { const double ix = px - V0x, iy = py - V0y, iz = pz - V0z, ex = V0x - V2x, ey = V0y - V2y, ez = V0z - V2z;
    const double cxx = (iy * ez) - (iz * ey), cyy = (iz * ex) - (ix * ez), czz = (ix * ey) - (iy * ex);
    if ((((cxx * Nx) + (cyy * Ny)) + (czz * Nz)) < -DRT_EPS) return false; }
  { const double ix = px - bx_, iy = py - by_, iz = pz - bz_, ex = bx_ - V0x, ey = by_ - V0y, ez = bz_ - V0z;
    const double cxx = (iy * ez) - (iz * ey), cyy = (iz * ex) - (ix * ez), czz = (ix * ey) - (iy * ex);
    if ((((cxx * Nx) + (cyy * Ny)) + (czz * Nz)) < -DRT_EPS) return false; }
  { const double ix = px - V2x, iy = py - V2y, iz = pz - V2z, ex = V2x - bx_, ey = V2y - by_, ez = V2z - bz_;
    const double cxx = (iy * ez) - (iz * ey), cyy = (iz * ex) - (ix * ez), czz = (ix * ey) - (iy * ex);
    if ((((cxx * Nx) + (cyy * Ny)) + (czz * Nz)) < -DRT_EPS) return false; }
  rank = __ldg(reinterpret_cast<const int32_t*>(T) + 29);
  tOut = t; stOut = st; return true;
}
// ---------------------------------------------------------------------------------------------------------------
// The one descent through a fast BVH (FP32 pre-test), closest hit and any hit.
// Almost every box decision is far from its boundary, so it is taken in FP32 on a 64-byte mirror of the node (FNode32: 4 loads instead of 7)
// under a rigorous error bound, and only an undecidable box goes to the reference's own FP64 test (true divisions, out of line).  Bound: with
// u = 2^-24, b32 = fl(b), inv32 = fl(1/a), oi32 = fl(o/a) and t32 = fma(b32, inv32, -oi32) (one rounding),
//     |t32 - (b - o)/a| <= u (3 |b/a| + 2 |o/a|) (1 + O(u)),        |b| <= absMax (per BVH, per axis),
// and the reference's FP64 quotient is within 2.3e-16 (|b/a| + |o/a|) of the same real number.  M = 1.1 u max_axis (3 absMax + 2 |o|) |1/a|
// (+ a denormal floor) therefore bounds the error of every slab value of the ray; min / max are 1-Lipschitz, so near32 / far32 are within M of
// the reference's biggestMin / min(tMax).  A box is ACCEPTED when far32 - near32 > 2M and near32 > M (=> far > near and near > 0 in the
// reference's arithmetic), REJECTED when far32 - near32 < -2M or near32 < -M, otherwise undecided.  Rays whose reciprocals or products leave the
// comfortable float range get M = +inf: every comparison fails and every box takes the exact test -- this is how the generic kernels serve an
// axis-parallel ray (a reciprocal of +-inf).  Entry times only order and prune (conservative lower bound near32 - M); triangles are always
// tested in FP64.
struct Lean32 { float ix, iy, iz, ox, oy, oz, M, M2; };
__device__ __forceinline__ Lean32 makeLean32(const FBvh& B, double ox, double oy, double oz, const D3& inv) {      // inv = rayInv() of the ray the boxes are tested with
  const double ix = inv.x, iy = inv.y, iz = inv.z; Lean32 L;
  L.ix = (float)ix; L.iy = (float)iy; L.iz = (float)iz; L.ox = (float)(ox * ix); L.oy = (float)(oy * iy); L.oz = (float)(oz * iz);
  const double ex = (3.0 * B.absMax[0] + 2.0 * fabs(ox)) * fabs(ix), ey = (3.0 * B.absMax[1] + 2.0 * fabs(oy)) * fabs(iy), ez = (3.0 * B.absMax[2] + 2.0 * fabs(oz)) * fabs(iz);
  double m = ex > ey ? ex : ey; m = ez > m ? ez : m;
  const double lim = 1e15; const bool sane = fabs(ix) < lim && fabs(iy) < lim && fabs(iz) < lim && fabs(ix) > 1e-15 && fabs(iy) > 1e-15 && fabs(iz) > 1e-15 &&
                                             B.absMax[0] < lim && B.absMax[1] < lim && B.absMax[2] < lim && m < 1e30;
  L.M = sane ? __double2float_ru(m * (1.1 * 5.9604644775390625e-8) + 1e-30) : __int_as_float(0x7f800000);
  L.M2 = 2.0f * L.M; return L;
}
// 1 accepted / 0 rejected / -1 undecided; nearOut = near32 (within M of the reference's entry t)
__device__ __forceinline__ int leanBox32(float mnx, float mny, float mnz, float mxx, float mxy, float mxz, const Lean32& L, bool stdBox, float& nearOut) {
  const float t1x = __fmaf_rn(mnx, L.ix, -L.ox), t2x = __fmaf_rn(mxx, L.ix, -L.ox), t1y = __fmaf_rn(mny, L.iy, -L.oy), t2y = __fmaf_rn(mxy, L.iy, -L.oy), t1z = __fmaf_rn(mnz, L.iz, -L.oz), t2z = __fmaf_rn(mxz, L.iz, -L.oz);
  float near_ = fmaxf(fmaxf(fminf(t1x, t2x), fminf(t1y, t2y)), fminf(t1z, t2z));
  const float far_ = fminf(fminf(fmaxf(t1x, t2x), fmaxf(t1y, t2y)), fmaxf(t1z, t2z));
  if (stdBox) { near_ = fmaxf(near_, 0.0f); nearOut = near_; const float gap = far_ - near_; return gap > L.M2 ? 1 : (gap < -L.M2 ? 0 : -1); }      // conventional: far >= max(near, 0)
  nearOut = near_; const float gap = far_ - near_;
  if (gap > L.M2 && near_ > L.M) return 1;
  if (gap < -L.M2 || near_ < -L.M) return 0;
  return -1;
}
// tScale (<= 1): lower bound of |ba| when the triangles see the NORMALISED direction of a ray whose box-space direction ba is shorter than unit
// length (an instance that enlarges its mesh, SURVEY Q7): a box entered at te (box units) is entered at te |ba| in triangle units, so a subtree
// may be skipped against the best hit only if te * tScale >= bestT.  1 when |ba| >= 1 (te itself is then the conservative bound).
__device__ __forceinline__ float leanScale(double len2) { return len2 >= 1.0 ? 1.0f : __double2float_rd(sqrt(len2)) * 0.999999f; }
// Closest hit inside one fast BVH (root box already accepted by the caller).  (bo, ba, binv) is the ray the boxes are tested with, (to, td) the
// ray the triangles are tested with (see SURVEY Q7 for why they can differ).  Result: the minimum-t hit over every leaf whose chain of boxes is
// accepted -- the set the reference's left-first recursion searches; equal-t candidates resolve to the lower reference rank, i.e. the reference's
// visiting order.  It is written to `out` only when strictly closer than `bound`.  Returns 1 hit / 0 miss / -1 the CAP-entry stack overflowed
// (the caller defers the ray to the generic kernel or flags a device error).  tc (counter builds): node visits (two boxes each), triangle tests.
// Loop shape ("while-while"): every lane first descends inner nodes until it HOLDS A LEAF (or is finished), then the warp tests triangles
// together -- the triangle test is the expensive, divergence-prone part (measured: 11.6 of 32 lanes active in the one-loop form).
// Stack entry: x = child reference (>= 0 inner node, < 0: ~tri-leaf code), y = bits of the lower bound of its box-entry t.  (The stack array and
// its scalar state are separate variables: a struct holding a dynamically indexed array lives in local memory as a whole, and `sp` would be
// re-loaded and re-stored on every push and pop.)
template <int CAP, bool ANY_DIR = false>
__device__ DRT_LEAN_INLINE int leanClosest32(const DScene& S, const FBvh& B, const D3 bo, const D3 ba, const D3 binv, const D3 to, const D3 td, const D3 rawDir, Hit& out, const double bound,
                                             const float tScale = 1.0f, TraceCounters* tc = nullptr) {
  const Lean32 L = makeLean32(B, bo.x, bo.y, bo.z, binv);
  const bool stdBox = S.accelMode == 2;
  uint2 stkE[CAP]; int sp = 0; bool overflow = false;
  // bestTf = bestT / tScale rounded UP: te_lb >= bestTf implies te * tScale >= bestT (the callers without a bound fold this to +inf)
  double bestT = bound; float bestTf = bound < DRT_DMAX ? __fdiv_ru(__double2float_ru(bound), tScale) : __int_as_float(0x7f800000);
  int bestTri = -1, bestRank = 0x7fffffff, bestSt = 0;
  int32_t ref = B.fastRoot; bool alive = true;
  auto popNext = [&]() { alive = false; while (sp > 0) { const uint2 e = stkE[--sp]; if (__uint_as_float(e.y) < bestTf) { ref = (int32_t)e.x; alive = true; break; } } };
  auto exact = [&](const FNode* nd, int side) -> float {     // undecided box: the reference's own test; returns a lower bound of the entry t, or -1 (rejected)
    const double* b6 = reinterpret_cast<const double*>(nd) + 6 * side;
    const double te = stdBox ? boxStdEntry<ANY_DIR>(b6, bo.x, bo.y, bo.z, ba.x, ba.y, ba.z) : boxExactEntry(b6, bo.x, bo.y, bo.z, ba.x, ba.y, ba.z);
    return (stdBox ? te >= 0 : te > 0) ? __double2float_rd(te) : -1.0f;
  };
  while (true) {
    // [sass:node-begin]  (tools/sass_model.py attributes the SASS between these markers to "one node visit")
    while (alive && ref >= 0) {
      const float4* q = reinterpret_cast<const float4*>(S.fnodes32 + ref);
      const float4 q0 = __ldg(q), q1 = __ldg(q + 1), q2 = __ldg(q + 2); const int4 lk = __ldg(reinterpret_cast<const int4*>(q) + 3);
      if (tc) tc->box += 2;
      float teL, teR;
      const int ql = leanBox32(q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, L, stdBox, teL), qr = leanBox32(q1.z, q1.w, q2.x, q2.y, q2.z, q2.w, L, stdBox, teR);
      bool hl = ql > 0, hr = qr > 0;
      if (ql >= 0) teL -= L.M; else { teL = exact(S.fnodes + ref, 0); hl = teL >= 0; }
      if (qr >= 0) teR -= L.M; else { teR = exact(S.fnodes + ref, 1); hr = teR >= 0; }
      hl = hl && teL < bestTf; hr = hr && teR < bestTf;
      const int32_t cl = childRef(lk.x, lk.z), cr = childRef(lk.y, lk.w);
      if (hl && hr) {
        const bool rightFirst = teR < teL;
        if (sp < CAP) stkE[sp++] = make_uint2((uint32_t)(rightFirst ? cl : cr), __float_as_uint(rightFirst ? teL : teR)); else overflow = true;
        ref = rightFirst ? cr : cl;
      } else if (hl) ref = cl;
      else if (hr) ref = cr;
      else popNext();
    }
    // [sass:node-end]
    if (!alive) break;
    // [sass:leaf-begin]
    {
      const int code = ~ref, cnt = code & 7, first = code >> 3;
      for (int i = 0; i < cnt; ++i) {
        double t; int st; int32_t rank; if (tc) ++tc->prim;
        if (leanTri(S.tris + first + i, to.x, to.y, to.z, td.x, td.y, td.z, bestT, t, st, rank) && (t < bestT || rank < bestRank)) { bestT = t; bestTf = __fdiv_ru(__double2float_ru(t), tScale); bestTri = first + i; bestRank = rank; bestSt = st; }
      }
    }
    // [sass:leaf-end]
    popNext();
  }
  if (overflow) return -1;
  if (bestTri < 0 || !(bestT < bound)) return 0;
  out.t = bestT; out.prim = S.tris[bestTri].prim; out.arg0 = 0; out.arg1 = 0; out.state = bestSt; out.hitXform = B.triHitXform; out.shaderOverride = -1; out.inst = -1; out.pad0 = 0;
  out.loc = d3((td.x * bestT) + to.x, (td.y * bestT) + to.y, (td.z * bestT) + to.z); out.rawDir = rawDir; return 1;
}
// Any hit inside one fast BVH: (dist - t) > eps for a triangle, every box on the way accepted with (dist - entry) > eps.  Rays and results as leanClosest32.
template <int CAP, bool ANY_DIR = false>
__device__ DRT_LEAN_INLINE int leanShadow32(const DScene& S, const FBvh& B, const D3 bo, const D3 ba, const D3 binv, const D3 to, const D3 td, double dist, TraceCounters* tc = nullptr) {
  const Lean32 L = makeLean32(B, bo.x, bo.y, bo.z, binv);
  const bool stdBox = S.accelMode == 2;
  // (dist - entry) > eps decided on near32 when it clears the bound: entry < dist - eps - M  /  entry > dist - eps + M
  const float accBelow = __double2float_rd((dist - DRT_EPS) - (double)L.M * 1.000001), rejAbove = __double2float_ru((dist - DRT_EPS) + (double)L.M * 1.000001);
  int32_t stkE[CAP]; int sp = 0; bool overflow = false;
  int32_t ref = B.fastRoot; bool alive = true, found = false;
  auto accept = [&](int q, float te, const FNode* nd, int side) {
    if (q == 0) return false;
    if (q > 0) { if (te < accBelow) return true; if (te > rejAbove) return false; }
    const double* b6 = reinterpret_cast<const double*>(nd) + 6 * side;
    const double tx = stdBox ? boxStdEntry<ANY_DIR>(b6, bo.x, bo.y, bo.z, ba.x, ba.y, ba.z) : boxExactEntry(b6, bo.x, bo.y, bo.z, ba.x, ba.y, ba.z);
    return (stdBox ? tx >= 0 : tx > 0) && (dist - tx) > DRT_EPS;
  };
  while (true) {
    // [sass:node-begin]  (tools/sass_model.py attributes the SASS between these markers to "one node visit")
    while (alive && ref >= 0) {
      const float4* q = reinterpret_cast<const float4*>(S.fnodes32 + ref);
      const float4 q0 = __ldg(q), q1 = __ldg(q + 1), q2 = __ldg(q + 2); const int4 lk = __ldg(reinterpret_cast<const int4*>(q) + 3);
      if (tc) tc->box += 2;
      float teL, teR;
      const int ql = leanBox32(q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, L, stdBox, teL), qr = leanBox32(q1.z, q1.w, q2.x, q2.y, q2.z, q2.w, L, stdBox, teR);
      const bool hl = accept(ql, teL, S.fnodes + ref, 0), hr = accept(qr, teR, S.fnodes + ref, 1);
      const int32_t cl = childRef(lk.x, lk.z), cr = childRef(lk.y, lk.w);
      if (hl && hr) { if (sp < CAP) stkE[sp++] = cr; else overflow = true; ref = cl; }
      else if (hl) ref = cl;
      else if (hr) ref = cr;
      else if (sp > 0) ref = stkE[--sp];
      else alive = false;
    }
    // [sass:node-end]
    if (!alive) break;
    // [sass:leaf-begin]
    {
      const int code = ~ref, cnt = code & 7, first = code >> 3;
      for (int i = 0; i < cnt; ++i) {
        double t; int st; int32_t rank; if (tc) ++tc->prim;
        if (leanTri(S.tris + first + i, to.x, to.y, to.z, td.x, td.y, td.z, DRT_DMAX, t, st, rank) && (dist - t) > DRT_EPS) { found = true; break; }
      }
    }
    // [sass:leaf-end]
    if (found) break;
    if (sp > 0) ref = stkE[--sp]; else alive = false;
  }
  if (found) return 1;
  return overflow ? -1 : 0;
}
__device__ __forceinline__ bool sameRay(const Ray& trans, const Ray& r) { return trans.o.x == r.o.x && trans.o.y == r.o.y && trans.o.z == r.o.z && trans.a.x == r.d.x && trans.a.y == r.d.y && trans.a.z == r.d.z; }

#define DRT_STACK 48
struct Frame { int32_t node; double tL; };     // node >= 0: "after left" of that node; node == -1: "after right", tL saved

// ---------------------------------------------------------------------------------------------------------------
// closest hit.  Every function returns 1 (hit), 0 (miss) or -1 (this kernel variant cannot serve the ray: defer it)
// ---------------------------------------------------------------------------------------------------------------
template <int F, int LVL>
__device__ __forceinline__ int accelClosestImpl(const DScene& S, int kind, int idx, Ray& _ray, const Ray& trans, int transXf, double time, Hit& out, TraceCounters* tc, double bound);
// the generic variant keeps one outlined copy per level (code size); the lean variants inline everything so that ray / hit records stay in registers
template <int F, int LVL>
__device__ __noinline__ int accelClosestOut(const DScene& S, int kind, int idx, Ray& _ray, const Ray& trans, int transXf, double time, Hit& out, TraceCounters* tc, double bound) { return accelClosestImpl<F, LVL>(S, kind, idx, _ray, trans, transXf, time, out, tc, bound); }
template <int F, int LVL>
__device__ __forceinline__ int accelClosest(const DScene& S, int kind, int idx, Ray& _ray, const Ray& trans, int transXf, double time, Hit& out, TraceCounters* tc, double bound) {
  if constexpr (F == TF_ALL) return accelClosestOut<F, LVL>(S, kind, idx, _ray, trans, transXf, time, out, tc, bound);
  else return accelClosestImpl<F, LVL>(S, kind, idx, _ray, trans, transXf, time, out, tc, bound);
}

// myGeomList.traverseStruct: every child gets a fresh transform of `_ray`; first strictly smaller t wins;
// the winner's CTM becomes list.CTM x child.CTM (child.hitXform).
// children of one mesh normally share one CTM: the transformed ray is a pure function of (_ray, xform), so it is kept
struct XfCache { int xf; Ray r; };
__device__ __forceinline__ const Ray& xfRayCached(const DScene& S, Ray& _ray, int xf, XfCache& xc) {
  if (xc.xf != xf) { xc.r = xfRay(_ray, S.xforms[xf].inv); xc.xf = xf; }
  return xc.r;
}
template <int F, int LVL>
__device__ __forceinline__ double leafClosest(const DScene& S, int listIdx, Ray& _ray, double time, Hit& res, TraceCounters* tc, XfCache& xc, bool& defer, double bound) {
  const FList L = S.lists[listIdx];
  double clsT = bound;
  for (int i = 0; i < L.childCount; ++i) {
    const FObjRef c = S.children[L.childStart + i];
    Ray r = xfRayCached(S, _ray, c.xform, xc);
    if (c.kind == OK_PRIM) {
      PHit ph; if (tc) ++tc->prim;
      if (primTest(S, c.idx, r, time, ph) && ph.t < clsT) { clsT = ph.t; takeHit(S, res, ph, c.idx, r, _ray.d, c.hitXform); res.pad0 += 2 * (L.childStart + i + 1); }
    } else {   // instance: the already transformed ray is forwarded as both rays (mySceneObject.java:123-127)
      const FInstance I = S.instances[c.idx];
      if (I.baseKind == OK_PRIM) {
        PHit ph; if (tc) ++tc->prim;
        if (primTest(S, I.baseIdx, r, time, ph) && ph.t < clsT) { clsT = ph.t; takeHit(S, res, ph, I.baseIdx, r, r.d, c.hitXform); res.pad0 += 2 * (L.childStart + i + 1); if (I.shader >= 0) res.shaderOverride = I.shader; res.inst = I.serial; }
      } else if constexpr (LVL == 1) {
        if constexpr (!(F & TF_LITERAL1)) { defer = true; return clsT; }
        else {
          Hit h; hitReset(h);
          const int got = accelClosest<F, 2>(S, I.baseKind, I.baseIdx, r, r, -1, time, h, tc, DRT_DMAX);
          if (got < 0) { defer = true; return clsT; }
          if (got && h.t < clsT) {
            clsT = h.t; res.t = h.t; res.prim = h.prim; res.arg0 = h.arg0; res.arg1 = h.arg1; res.state = h.state; res.loc = h.loc; res.rawDir = h.rawDir;
            res.hitXform = c.hitXform; res.shaderOverride = (I.shader >= 0) ? I.shader : h.shaderOverride; res.inst = (h.inst < 0) ? I.serial : h.inst;
          }
        }
      }
    }
  }
  return clsT;
}

// myAccelStruct.intersectCheck (root gate) + myBVH.traverseStruct, iteratively.
// Semantics of the recursion kept exactly: left subtree first; right subtree only if its box is hit and
// (left found nothing or right-entry t < left result t); result = left if left.t <= right.t.  Because every level
// combines with "min, left wins ties", the overall winner is the DFS-first minimum over all visited leaves; the
// per-subtree minima needed for the pruning decisions live on an explicit frame stack.
template <int F, int LVL>
__device__ __forceinline__ int accelClosestImpl(const DScene& S, int kind, int idx, Ray& _ray, const Ray& trans, int transXf, double time, Hit& out, TraceCounters* tc, double bound) {
  constexpr bool LITERAL = (LVL == 1) ? ((F & TF_LITERAL1) != 0) : ((F & TF_LEVEL2) != 0);      // literal recursion compiled in at this level?
  const D3 inv = rayInv(trans);
  if (kind == OK_LIST) {
    const FList& L = S.lists[idx];
    if (tc) ++tc->box;
    if (!boxHit(L.bmin, L.bmax, trans, inv)) return 0;
    XfCache xc; xc.xf = -1; bool defer = false;
    double t = leafClosest<F, LVL>(S, idx, _ray, time, out, tc, xc, defer, bound);
    if (defer) return -1;
    return t < bound ? 1 : 0;
  }
  const FBvh& B = S.bvhs[idx];
  if (tc) ++tc->box;
  if (!boxHit(B.bmin, B.bmax, trans, inv)) return 0;
  if (S.accelMode != 0 && B.fast != 0) {
    const double len2 = _ray.norm ? 1.0 : dot3(_ray.d, _ray.d);      // < 1 through an instance that enlarges its mesh: the search scales its bound (leanScale)
    if (len2 > 1e-200) {
      // what every leaf child of this mesh would be tested with.  getTransformedRay is a pure function of (ray, CTM) once the source direction is
      // unit length, so when `trans` was formed from this very ray with the triangles' own CTM the two rays are the same bits: nothing to recompute
      const bool sameXf = _ray.norm && transXf == B.triXform;
      const Ray r = sameXf ? trans : xfRay(_ray, S.xforms[B.triXform].inv);
      if constexpr (F == TF_ALL) {
        const int got = leanClosest32<DRT_FSTACK, true>(S, B, trans.o, trans.a, inv, r.o, r.d, _ray.d, out, bound, leanScale(len2), tc);
        if (got < 0) { flagError(DEV_ERR_INCOMPLETE); return 0; }
        return got;
      } else {
        // the lean kernels defer axis-parallel rays.  One instantiation per lean kernel (one traversal stack in its frame): scenes with instanced
        // meshes need the two-ray form (which gives the same bits when both rays coincide), flat scenes test boxes and triangles with the same ray
        // and defer the rest
        const bool one = sameXf || sameRay(trans, r);
        if (regularDir(trans.a)) {
          if constexpr ((F & TF_LITERAL1) != 0) return leanClosest32<DRT_LSTACK>(S, B, trans.o, trans.a, inv, r.o, r.d, _ray.d, out, bound, leanScale(len2));
          else { if (!one) return -1; return leanClosest32<DRT_LSTACK>(S, B, trans.o, trans.a, inv, trans.o, trans.a, _ray.d, out, bound); }      // flat scenes: one ray, one register set
        }
      }
      return -1;
    }
  }
  if constexpr (!LITERAL) return -1;
  else {
  XfCache xc; xc.xf = -1; bool defer = false;
  Hit& best = out; hitReset(best);
  Hit leaf; hitReset(leaf);
  Frame stack[DRT_STACK]; int sp = 0;
  int32_t node = B.root; double tCur = DRT_DMAX;
  while (true) {
    bool ret = false;
    int32_t afterLeftOf = -1;
    if (node < 0) {                    // leaf
      tCur = leafClosest<F, LVL>(S, ~node, _ray, time, leaf, tc, xc, defer, DRT_DMAX);
      if (defer) return -1;
      if (tCur < best.t) { best.t = leaf.t; best.prim = leaf.prim; best.arg0 = leaf.arg0; best.arg1 = leaf.arg1; best.state = leaf.state; best.hitXform = leaf.hitXform;
        best.shaderOverride = leaf.shaderOverride; best.inst = leaf.inst; best.loc = leaf.loc; best.rawDir = leaf.rawDir; }
      ret = true;
    } else {
      const FNode& N = S.nodes[node];
      if (tc) ++tc->box;
      if (sp >= DRT_STACK) flagError(DEV_ERR_INCOMPLETE);
      if (boxHit(N.lmin, N.lmax, trans, inv) && sp < DRT_STACK) { stack[sp].node = node; stack[sp].tL = 0; ++sp; node = N.left; tCur = DRT_DMAX; continue; }
      tCur = DRT_DMAX; afterLeftOf = node;
    }
    while (true) {
      if (afterLeftOf >= 0) {          // left subtree of `afterLeftOf` finished with tCur
        const FNode& N = S.nodes[afterLeftOf];
        if (tc) ++tc->box;
        if (boxHitBefore(N.rmin, N.rmax, trans, inv, tCur) && sp < DRT_STACK) { stack[sp].node = -1; stack[sp].tL = tCur; ++sp; node = N.right; tCur = DRT_DMAX; ret = false; break; }
        afterLeftOf = -1; ret = true;  // result of this node = tL (an untraversed right box can never win: te >= tL)
      }
      if (ret) {
        if (sp == 0) return best.t < DRT_DMAX ? 1 : 0;
        --sp;
        if (stack[sp].node >= 0) { afterLeftOf = stack[sp].node; continue; }
        double tL = stack[sp].tL; tCur = (tL <= tCur) ? tL : tCur;       // min, left wins ties
        continue;
      }
    }
  }
  }
}

// myScene.findClosestRayHit: linear scan of the top-level list, first-inserted wins among equal t.
// The accel searches take `bound`: they write their winner to the record they are given only if it is strictly closer than bound -- the same
// decision as "h.t < best.t" on a separate record.  The flat lean variants (no literal recursion: every search they reach honours bound) pass
// `best` itself, so a single Hit lives across the BVH walk instead of two, and they carry only the winner's key across it: which top-level
// object (wTop) and, in best.pad0, which list child produced it.  Its hit point and recorded direction are formed once, after the loop, from
// the same transformed ray the winning test used: getTransformedRay is a pure function of (unit-length ray, CTM), so the recomputed ray has
// the bits the loop had.
template <int F>
__device__ __forceinline__ int closestHitT(const DScene& S, Ray& ray, double time, Hit& best, TraceCounters* tc) {
  constexpr bool IN_PLACE = (F & TF_LITERAL1) == 0;
  hitReset(best);
  Hit h; if constexpr (!IN_PLACE) hitReset(h);
  Ray tr; int trXf = -1;        // consecutive top-level objects often share one CTM (a polygon soup read under one transform): the transformed
                                // ray is a pure function of (ray, CTM), and `ray` is already unit length here, so it is formed once per run
  int wTop = -1;
  for (int i = 0; i < S.g.numTop; ++i) {
    const FObjRef o = S.top[i];
    if (o.xform != trXf || o.kind != OK_PRIM) { tr = xfRay(ray, S.xforms[o.xform].inv); trXf = (o.kind == OK_PRIM) ? o.xform : -1; }
    if (o.kind == OK_PRIM) {
      PHit ph; if (tc) ++tc->prim;
      const int triIdx = (S.accelMode != 0) ? S.prims[o.idx].pad0 : -1;      // packed record of a plain top-level triangle (fast modes)
      if (triIdx >= 0) {
        int32_t rank; ph.arg0 = 0; ph.arg1 = 0; ph.boxRaw = 0;
        if (leanTri(S.tris + triIdx, tr.o.x, tr.o.y, tr.o.z, tr.d.x, tr.d.y, tr.d.z, best.t, ph.t, ph.state, rank) && ph.t < best.t) { takeHit(S, best, ph, o.idx, tr, ray.d, o.xform); wTop = i; }
      } else if (primTest(S, o.idx, tr, time, ph) && ph.t < best.t) { takeHit(S, best, ph, o.idx, tr, ray.d, o.xform); wTop = i; }
    } else {
      int got; int shader = -1, serial = -1;
      if (o.kind == OK_INSTANCE) {
        const FInstance I = S.instances[o.idx]; shader = I.shader; serial = I.serial;
        if (I.baseKind == OK_PRIM) {
          PHit ph; if (tc) ++tc->prim;
          if (primTest(S, I.baseIdx, tr, time, ph) && ph.t < best.t) { takeHit(S, best, ph, I.baseIdx, tr, tr.d, o.xform); if (shader >= 0) best.shaderOverride = shader; best.inst = serial; wTop = i; }
          continue;
        }
        if constexpr (IN_PLACE) got = accelClosest<F, 1>(S, I.baseKind, I.baseIdx, tr, tr, -1, time, best, tc, best.t);
        else got = accelClosest<F, 1>(S, I.baseKind, I.baseIdx, tr, tr, -1, time, h, tc, DRT_DMAX);
      } else if constexpr (IN_PLACE) got = accelClosest<F, 1>(S, o.kind, o.idx, ray, tr, o.xform, time, best, tc, best.t);
      else got = accelClosest<F, 1>(S, o.kind, o.idx, ray, tr, o.xform, time, h, tc, DRT_DMAX);
      if (got < 0) return -1;
      if constexpr (IN_PLACE) {
        if (got) { if (shader >= 0) best.shaderOverride = shader; if (serial >= 0 && best.inst < 0) best.inst = serial; wTop = i; }
      } else if (got && h.t < best.t) {
        best.t = h.t; best.prim = h.prim; best.arg0 = h.arg0; best.arg1 = h.arg1; best.state = h.state; best.hitXform = h.hitXform; best.loc = h.loc; best.rawDir = h.rawDir;
        best.shaderOverride = (shader >= 0) ? shader : h.shaderOverride; best.inst = (serial >= 0 && h.inst < 0) ? serial : h.inst;
      }
    }
  }
  if constexpr (IN_PLACE) {
    best.loc = d3(0, 0, 0); best.rawDir = d3(0, 0, 0);
    if (wTop >= 0) {
      const FObjRef o = S.top[wTop];
      Ray tr0 = xfRay(ray, S.xforms[o.xform].inv);
      const int child = (best.pad0 >> 1) - 1; const bool boxRaw = (best.pad0 & 1) != 0;
      Ray rt = tr0; D3 raw;
      if (child >= 0) {           // primitive of a list (leafClosest): the list's ray -- renormalised in place through an instance -- under the child's CTM
        Ray& src = (o.kind == OK_INSTANCE) ? tr0 : ray;
        const FObjRef c = S.children[child];
        rt = xfRay(src, S.xforms[c.xform].inv);
        raw = (c.kind == OK_PRIM) ? src.d : rt.d;
      } else if (o.kind == OK_INSTANCE) {
        raw = (S.instances[o.idx].baseKind == OK_PRIM) ? tr0.d : norm3(tr0.d);    // instanced mesh: the lean search saw the renormalised ray
      } else raw = ray.d;
      best.loc = pointOnRay(rt, best.t);
      best.rawDir = boxRaw ? xfVector(S.xforms[S.prims[best.prim].xform].m, rt.d) : raw;
    }
  }
  return best.t < DRT_DMAX ? 1 : 0;
}
__device__ __forceinline__ bool closestHit(const DScene& S, Ray& ray, double time, Hit& best, TraceCounters* tc) { return closestHitT<TF_ALL>(S, ray, time, best, tc) > 0; }


// ---------------------------------------------------------------------------------------------------------------
// any hit (shadow rays): hit AND (distToLight - t) > eps.  The BVH form never tests its root box; every list
// (top-level or BVH leaf) gates on its own box with the same rule (SURVEY Q1b, Q19).  1 / 0 / -1 as above.
// ---------------------------------------------------------------------------------------------------------------
template <int F, int LVL>
__device__ __forceinline__ int accelShadowImpl(const DScene& S, int kind, int idx, Ray& _ray, const Ray& trans, int transXf, double time, double dist, TraceCounters* tc);
template <int F, int LVL>
__device__ __noinline__ int accelShadowOut(const DScene& S, int kind, int idx, Ray& _ray, const Ray& trans, int transXf, double time, double dist, TraceCounters* tc) { return accelShadowImpl<F, LVL>(S, kind, idx, _ray, trans, transXf, time, dist, tc); }
template <int F, int LVL>
__device__ __forceinline__ int accelShadow(const DScene& S, int kind, int idx, Ray& _ray, const Ray& trans, int transXf, double time, double dist, TraceCounters* tc) {
  if constexpr (F == TF_ALL) return accelShadowOut<F, LVL>(S, kind, idx, _ray, trans, transXf, time, dist, tc);
  else return accelShadowImpl<F, LVL>(S, kind, idx, _ray, trans, transXf, time, dist, tc);
}

template <int F, int LVL>
__device__ __forceinline__ int listShadow(const DScene& S, int listIdx, Ray& _ray, const Ray& trans, const D3& inv, double time, double dist, TraceCounters* tc, XfCache& xc) {
  const FList L = S.lists[listIdx];
  if (tc) ++tc->box;
  if (!boxAcceptShadow(L.bmin, L.bmax, trans, inv, dist)) return 0;
  for (int i = 0; i < L.childCount; ++i) {
    const FObjRef c = S.children[L.childStart + i];
    Ray r = xfRayCached(S, _ray, c.xform, xc);
    PHit h;
    if (c.kind == OK_PRIM) { if (tc) ++tc->prim; if (primTest(S, c.idx, r, time, h) && (dist - h.t) > DRT_EPS) return 1; }
    else {
      const FInstance I = S.instances[c.idx];
      if (I.baseKind == OK_PRIM) { if (tc) ++tc->prim; if (primTest(S, I.baseIdx, r, time, h) && (dist - h.t) > DRT_EPS) return 1; }
      else if constexpr (LVL == 1) {
        if constexpr (!(F & TF_LITERAL1)) return -1;
        else { const int got = accelShadow<F, 2>(S, I.baseKind, I.baseIdx, r, r, -1, time, dist, tc); if (got != 0) return got; }
      }
    }
  }
  return 0;
}
// Shadow rays through an INSTANCE TREE in the lean kernels: the walk of accelShadowImpl's literal loop + listShadow below, reorganised so that the
// lanes of a warp do their heavy work together.  Each lane advances its own walk in small steps (phase A: cheap node / pop steps until it stands
// at a leaf child, then the child step -- instance transform -- together) until it HOLDS AN INSTANCED MESH TO SEARCH; the lanes then search their
// meshes side by side in ONE call of the lean mesh traversal (phase B).  No ray's sequence of tests changes; measured on p3_t11_sierp 4K/16 spp:
// k_light 1067 -> 848 ms.  (The same reorganisation of the closest-hit walk, pooling the searches over the block, and persistent lanes that
// fetch new rays were all measured and lost or tied: profiles/r2_tuning.md.)
template <int F>
__device__ __forceinline__ int instTreeShadow(const DScene& S, const FBvh& B, Ray& _ray, const Ray& trans, const D3& inv, double time, double dist) {
  enum { M_VISIT = 0, M_LEAF = 1, M_POP = 2 };
  XfCache xc; xc.xf = -1;
  int32_t stack[DRT_STACK]; int sp = 0; int32_t node = B.root;
  int mode = M_VISIT, li = 0, leafStart = 0, leafCount = 0, result = 0;
  bool done = false, pending = false;
  int32_t pBvh = 0; D3 pbo = d3(0, 0, 0), pba = pbo, pinv = pbo, pto = pbo, ptd = pbo;
  while (!done) {
    while (!done && !pending) {
      while (!done && mode != M_LEAF) {       // cheap steps until every lane stands at a leaf child
      if (mode == M_VISIT) {
        if (node < 0) {
          const FList& L = S.lists[~node];
          if (!boxAcceptShadow(L.bmin, L.bmax, trans, inv, dist)) mode = M_POP;
          else { leafStart = L.childStart; leafCount = L.childCount; li = 0; mode = M_LEAF; }
        } else {
          const FNode& N = S.nodes[node];
          const bool hl = boxAcceptShadow(N.lmin, N.lmax, trans, inv, dist), hr = boxAcceptShadow(N.rmin, N.rmax, trans, inv, dist);
          if (hl) { if (hr) { if (sp < DRT_STACK) stack[sp++] = N.right; else flagError(DEV_ERR_INCOMPLETE); } node = N.left; }
          else if (hr) node = N.right;
          else mode = M_POP;
        }
      } else {
        if (sp == 0) { result = 0; done = true; }
        else { node = stack[--sp]; mode = M_VISIT; }
      }
      }
      if (!done) {
        if (li >= leafCount) mode = M_POP;
        else {
          const FObjRef c = S.children[leafStart + li]; ++li;
          Ray r = xfRayCached(S, _ray, c.xform, xc);
          PHit h;
          if (c.kind == OK_PRIM) { if (primTest(S, c.idx, r, time, h) && (dist - h.t) > DRT_EPS) { result = 1; done = true; } }
          else {
            const FInstance I = S.instances[c.idx];
            if (I.baseKind == OK_PRIM) { if (primTest(S, I.baseIdx, r, time, h) && (dist - h.t) > DRT_EPS) { result = 1; done = true; } }
            else if (I.baseKind == OK_BVH) {                // accelShadowImpl<F, 2>: no root gate (SURVEY Q19)
              const FBvh& B2 = S.bvhs[I.baseIdx];
              if (!(S.accelMode != 0 && B2.fast != 0) || !regularDir(r.a)) { result = -1; done = true; }
              else {
                const D3 inv2 = rayInv(r);
                const Ray r2 = xfRay(r, S.xforms[B2.triXform].inv);
                pending = true; pBvh = I.baseIdx; pbo = r.o; pba = r.a; pinv = inv2; pto = r2.o; ptd = r2.d;
              }
            } else { const int got = accelShadow<F, 2>(S, I.baseKind, I.baseIdx, r, r, -1, time, dist, nullptr); if (got != 0) { result = got; done = true; } }
          }
        }
      }
    }
    if (pending) {                          // phase B: the lanes that hold a mesh search it side by side
      const int got = leanShadow32<DRT_LSTACK>(S, S.bvhs[pBvh], pbo, pba, pinv, pto, ptd, dist);
      if (got != 0) { result = got; done = true; }
      pending = false;
    }
  }
  return result;
}
template <int F, int LVL>
__device__ __forceinline__ int accelShadowImpl(const DScene& S, int kind, int idx, Ray& _ray, const Ray& trans, int transXf, double time, double dist, TraceCounters* tc) {
  constexpr bool LITERAL = (LVL == 1) ? ((F & TF_LITERAL1) != 0) : ((F & TF_LEVEL2) != 0);
  const D3 inv = rayInv(trans);
  XfCache xc; xc.xf = -1;
  if (kind == OK_LIST) return listShadow<F, LVL>(S, idx, _ray, trans, inv, time, dist, tc, xc);
  const FBvh& B = S.bvhs[idx];
  if (S.accelMode != 0 && B.fast != 0) {                              // any-hit does not depend on the visiting order
    const bool sameXf = _ray.norm && transXf == B.triXform;          // see accelClosestImpl
    const Ray r = sameXf ? trans : xfRay(_ray, S.xforms[B.triXform].inv);
    if constexpr (F == TF_ALL) {
      const int got = leanShadow32<DRT_FSTACK, true>(S, B, trans.o, trans.a, inv, r.o, r.d, dist, tc);
      if (got < 0) { flagError(DEV_ERR_INCOMPLETE); return 0; }
      return got;
    } else {
      const bool one = sameXf || sameRay(trans, r);
      if (regularDir(trans.a)) {
        if constexpr ((F & TF_LITERAL1) != 0) return leanShadow32<DRT_LSTACK>(S, B, trans.o, trans.a, inv, r.o, r.d, dist);
        else { if (!one) return -1; return leanShadow32<DRT_LSTACK>(S, B, trans.o, trans.a, inv, trans.o, trans.a, dist); }
      }
    }
    return -1;
  }
  if constexpr (!LITERAL) return -1;
  else if constexpr (F != TF_ALL && LVL == 1) return instTreeShadow<F>(S, B, _ray, trans, inv, time, dist);
  else {
  int32_t stack[DRT_STACK]; int sp = 0; int32_t node = B.root;
  while (true) {
    if (node < 0) { const int got = listShadow<F, LVL>(S, ~node, _ray, trans, inv, time, dist, tc, xc); if (got != 0) return got; }
    else {
      const FNode& N = S.nodes[node];
      if (tc) tc->box += 2;
      bool hl = boxAcceptShadow(N.lmin, N.lmax, trans, inv, dist);
      bool hr = boxAcceptShadow(N.rmin, N.rmax, trans, inv, dist);
      if (hl) { if (hr) { if (sp < DRT_STACK) stack[sp++] = N.right; else flagError(DEV_ERR_INCOMPLETE); } node = N.left; continue; }
      if (hr) { node = N.right; continue; }
    }
    if (sp == 0) return 0;
    node = stack[--sp];
  }
  }
}
template <int F>
__device__ __forceinline__ int anyHitT(const DScene& S, Ray& ray, double time, double dist, TraceCounters* tc) {
  Ray tr; int trXf = -1;
  for (int i = 0; i < S.g.numTop; ++i) {
    const FObjRef o = S.top[i];
    if (o.xform != trXf || o.kind != OK_PRIM) { tr = xfRay(ray, S.xforms[o.xform].inv); trXf = (o.kind == OK_PRIM) ? o.xform : -1; }
    PHit h;
    if (o.kind == OK_PRIM) {
      if (tc) ++tc->prim;
      const int triIdx = (S.accelMode != 0) ? S.prims[o.idx].pad0 : -1;
      if (triIdx >= 0) { int32_t rank; if (leanTri(S.tris + triIdx, tr.o.x, tr.o.y, tr.o.z, tr.d.x, tr.d.y, tr.d.z, DRT_DMAX, h.t, h.state, rank) && (dist - h.t) > DRT_EPS) return 1; }
      else if (primTest(S, o.idx, tr, time, h) && (dist - h.t) > DRT_EPS) return 1;
    }
    else if (o.kind == OK_INSTANCE) {
      const FInstance I = S.instances[o.idx];
      if (I.baseKind == OK_PRIM) { if (tc) ++tc->prim; if (primTest(S, I.baseIdx, tr, time, h) && (dist - h.t) > DRT_EPS) return 1; }
      else { const int got = accelShadow<F, 1>(S, I.baseKind, I.baseIdx, tr, tr, -1, time, dist, tc); if (got != 0) return got; }
    } else { const int got = accelShadow<F, 1>(S, o.kind, o.idx, ray, tr, o.xform, time, dist, tc); if (got != 0) return got; }
  }
  return 0;
}


}  // namespace drt
