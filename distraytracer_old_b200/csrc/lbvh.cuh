// GPU LBVH builder for the pure-triangle ("fast") BVHs: 30-bit Morton codes of the triangle-box centres, stable radix sort
// (dev_sort.cuh), clusters of <= 4 consecutive triangles as leaves, Karras-2012 hierarchy over the cluster codes, bottom-up refit that
// writes the final 128-byte nodes (both child boxes per node) directly.
//
// Performance-mode replacement of the reference's top-down median-split build, myBVH.addObjList / buildSortedObjAras
// (myGeomBase.java:338-386; O(N log^2 N) TreeMap re-sorting per node, one 4x4 inverse per node).  The triangle set is the one the
// reference tree holds (its dropped object, SURVEY Q2, is already absent from the packed records), the root-box gate stays the
// reference's (SURVEY Q1a), so primary-ray hit IDs are unchanged; see DESIGN.md for what cannot match (Q1b).
#pragma once
#include "dbuf.h"
#include "dev_sort.cuh"

namespace drt {

__device__ __forceinline__ uint32_t mortonExpand10(uint32_t v) { v &= 1023u; v = (v * 0x00010001u) & 0xFF0000FFu; v = (v * 0x00000101u) & 0x0F00F00Fu; v = (v * 0x00000011u) & 0xC30C30C3u; v = (v * 0x00000005u) & 0x49249249u; return v; }

struct LbvhBox { double mn[3], mx[3]; };

__global__ void k_lbvh_morton(const FTri* __restrict__ tris, int n, LbvhBox root, uint32_t* __restrict__ keys) {
  int i = blockIdx.x * blockDim.x + threadIdx.x; if (i >= n) return;
  const double* v = tris[i].v; uint32_t q[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const double lo = fmin(v[k], fmin(v[3 + k], v[6 + k])), hi = fmax(v[k], fmax(v[3 + k], v[6 + k])), c = 0.5 * (lo + hi);
    const double ext = root.mx[k] - root.mn[k]; double u = ext > 0 ? (c - root.mn[k]) / ext : 0.0; u = fmin(fmax(u * 1024.0, 0.0), 1023.0); q[k] = (uint32_t)u;
  }
  keys[i] = (mortonExpand10(q[0]) << 2) | (mortonExpand10(q[1]) << 1) | mortonExpand10(q[2]);
}
// sorted order -> packed records in place of the BVH's range (8 threads move one 128-byte triangle with 128-bit accesses)
__global__ void k_lbvh_gather(const FTri* __restrict__ src, const uint32_t* __restrict__ order, int n, FTri* __restrict__ dst) {
  long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; int i = (int)(t >> 3), c = (int)(t & 7); if (i >= n) return;
  reinterpret_cast<int4*>(dst + i)[c] = __ldg(reinterpret_cast<const int4*>(src + order[i]) + c);
}
// one leaf = up to 4 consecutive sorted triangles: conservative box (padded outward), Morton code of its first triangle
__global__ void k_lbvh_leaves(const FTri* __restrict__ sorted, const uint32_t* __restrict__ sortedKeys, int nTris, int nLeaves, LbvhBox* __restrict__ leafBox, uint32_t* __restrict__ leafCode) {
  int j = blockIdx.x * blockDim.x + threadIdx.x; if (j >= nLeaves) return;
  LbvhBox b; for (int k = 0; k < 3; ++k) { b.mn[k] = DRT_DMAX; b.mx[k] = -DRT_DMAX; }
  const int first = 4 * j, cnt = min(4, nTris - first);
  for (int i = 0; i < cnt; ++i) { const double* v = sorted[first + i].v; for (int p = 0; p < 3; ++p) for (int k = 0; k < 3; ++k) { b.mn[k] = fmin(b.mn[k], v[3 * p + k]); b.mx[k] = fmax(b.mx[k], v[3 * p + k]); } }
  for (int k = 0; k < 3; ++k) { b.mn[k] -= 1e-12 * fmax(1.0, fabs(b.mn[k])); b.mx[k] += 1e-12 * fmax(1.0, fabs(b.mx[k])); }
  leafBox[j] = b; leafCode[j] = sortedKeys[first];
}
// Karras 2012: internal node i of the radix tree over the (code, index) keys
__device__ __forceinline__ int lbvhDelta(const uint32_t* __restrict__ code, int n, int i, int j) {
  if (j < 0 || j >= n) return -1;
  const uint64_t a = ((uint64_t)code[i] << 32) | (uint32_t)i, b = ((uint64_t)code[j] << 32) | (uint32_t)j;
  return __clzll((long long)(a ^ b));
}
__global__ void k_lbvh_hierarchy(const uint32_t* __restrict__ code, int nLeaves, int2* __restrict__ child /*[n-1]: x=left y=right; >=0 internal, <0 ~leaf*/, int* __restrict__ parentInternal, int* __restrict__ parentLeaf) {
  int i = blockIdx.x * blockDim.x + threadIdx.x; if (i >= nLeaves - 1) return;
  const int d = (lbvhDelta(code, nLeaves, i, i + 1) - lbvhDelta(code, nLeaves, i, i - 1)) >= 0 ? 1 : -1;
  const int dMin = lbvhDelta(code, nLeaves, i, i - d);
  int lmax = 2; while (lbvhDelta(code, nLeaves, i, i + lmax * d) > dMin) lmax <<= 1;
  int l = 0; for (int t = lmax >> 1; t >= 1; t >>= 1) if (lbvhDelta(code, nLeaves, i, i + (l + t) * d) > dMin) l += t;
  const int j = i + l * d, dNode = lbvhDelta(code, nLeaves, i, j);
  int s = 0, t = l;
  do { t = (t + 1) >> 1; if (lbvhDelta(code, nLeaves, i, i + (s + t) * d) > dNode) s += t; } while (t > 1);
  const int gamma = i + s * d + min(d, 0);
  const int lo = min(i, j), hi = max(i, j);
  int2 c; c.x = (lo == gamma) ? ~gamma : gamma; c.y = (hi == gamma + 1) ? ~(gamma + 1) : (gamma + 1);
  child[i] = c;
  if (c.x >= 0) parentInternal[c.x] = i; else parentLeaf[~c.x] = i;
  if (c.y >= 0) parentInternal[c.y] = i; else parentLeaf[~c.y] = i;
  if (i == 0) parentInternal[0] = -1;
}
// bottom-up: the second thread to reach a node owns it, forms its box and writes the final node record
__global__ void k_lbvh_refit(int nLeaves, int nTris, int triBase, int nodeBase, const int2* __restrict__ child, const int* __restrict__ parentInternal, const int* __restrict__ parentLeaf,
                             const LbvhBox* __restrict__ leafBox, LbvhBox* nodeBox, unsigned int* flags, FNode* __restrict__ nodesOut) {
  int j = blockIdx.x * blockDim.x + threadIdx.x; if (j >= nLeaves) return;
  int cur = parentLeaf[j];
  while (cur >= 0) {
    __threadfence();
    if (atomicAdd(&flags[cur], 1u) == 0u) return;
    const int2 c = child[cur]; LbvhBox L, R;
    const volatile LbvhBox* nb = nodeBox;
    if (c.x < 0) L = leafBox[~c.x]; else for (int k = 0; k < 3; ++k) { L.mn[k] = nb[c.x].mn[k]; L.mx[k] = nb[c.x].mx[k]; }
    if (c.y < 0) R = leafBox[~c.y]; else for (int k = 0; k < 3; ++k) { R.mn[k] = nb[c.y].mn[k]; R.mx[k] = nb[c.y].mx[k]; }
    FNode N;
    for (int k = 0; k < 3; ++k) { N.lmin[k] = L.mn[k]; N.lmax[k] = L.mx[k]; N.rmin[k] = R.mn[k]; N.rmax[k] = R.mx[k]; }
    auto triCode = [&](int leaf) { const int first = 4 * leaf, cnt = min(4, nTris - first); return (int32_t)(((triBase + first) << 3) | cnt); };
    N.left = c.x >= 0 ? nodeBase + c.x : -1; N.right = c.y >= 0 ? nodeBase + c.y : -1;
    N.triL = c.x < 0 ? triCode(~c.x) : -1; N.triR = c.y < 0 ? triCode(~c.y) : -1; N.pad2[0] = N.pad2[1] = N.pad2[2] = N.pad2[3] = 0;
    nodesOut[cur] = N;
    LbvhBox U; for (int k = 0; k < 3; ++k) { U.mn[k] = fmin(L.mn[k], R.mn[k]); U.mx[k] = fmax(L.mx[k], R.mx[k]); }
    nodeBox[cur] = U;
    cur = parentInternal[cur];
  }
}

// host driver: rebuilds one BVH. `trisAll` is the device copy of the packed-triangle array (the BVH's range is re-ordered in place),
// nodesOut receives nLeaves-1 nodes whose child links are absolute (nodeBase + i). Returns the number of nodes written (0 = not rebuilt).
struct LbvhScratch {
  DBuf<uint32_t> keys[2], vals[2], hist, scan, leafCode; DBuf<unsigned int> flags; DBuf<FTri> tmp; DBuf<LbvhBox> leafBox, nodeBox; DBuf<int2> child; DBuf<int> parentI, parentL;
  void ensure(size_t n, cudaStream_t st) {
    for (int k = 0; k < 2; ++k) { keys[k].ensure(n, st); vals[k].ensure(n, st); }
    const long long nb = radixBlocks((long long)n);
    hist.ensure((size_t)256 * nb, st); scan.ensure((size_t)scanScratchWords(256 * nb), st);
    leafCode.ensure(n, st); flags.ensure(n, st); tmp.ensure(n, st); leafBox.ensure(n, st); nodeBox.ensure(n, st); child.ensure(n, st); parentI.ensure(n, st); parentL.ensure(n, st);
  }
};
static inline int lbvhBuild(FTri* trisAll, int triStart, int nTris, const double bmin[3], const double bmax[3], FNode* nodesOut, int nodeBase, LbvhScratch& sc, cudaStream_t st) {
  const int nLeaves = (nTris + 3) / 4; if (nLeaves < 2) return 0;
  sc.ensure((size_t)nTris, st);
  LbvhBox root; for (int k = 0; k < 3; ++k) { root.mn[k] = bmin[k]; root.mx[k] = bmax[k]; }
  FTri* range = trisAll + triStart;
  uint32_t* keys[2] = {sc.keys[0].p, sc.keys[1].p}; uint32_t* vals[2] = {sc.vals[0].p, sc.vals[1].p};
  k_lbvh_morton<<<(nTris + 255) / 256, 256, 0, st>>>(range, nTris, root, keys[0]); ++g_kernelLaunches;
  const int cur = radixSortPairs(keys, vals, nTris, 30, true, sc.hist.p, sc.scan.p, st);
  k_lbvh_gather<<<(unsigned)(((long long)nTris * 8 + 255) / 256), 256, 0, st>>>(range, vals[cur], nTris, sc.tmp.p); ++g_kernelLaunches;
  CK(cudaMemcpyAsync(range, sc.tmp.p, (size_t)nTris * sizeof(FTri), cudaMemcpyDeviceToDevice, st));
  k_lbvh_leaves<<<(nLeaves + 255) / 256, 256, 0, st>>>(range, keys[cur], nTris, nLeaves, sc.leafBox.p, sc.leafCode.p); ++g_kernelLaunches;
  k_lbvh_hierarchy<<<(nLeaves - 1 + 255) / 256, 256, 0, st>>>(sc.leafCode.p, nLeaves, sc.child.p, sc.parentI.p, sc.parentL.p); ++g_kernelLaunches;
  CK(cudaMemsetAsync(sc.flags.p, 0, (size_t)nLeaves * 4, st));
  k_lbvh_refit<<<(nLeaves + 255) / 256, 256, 0, st>>>(nLeaves, nTris, triStart, nodeBase, sc.child.p, sc.parentI.p, sc.parentL.p, sc.leafBox.p, sc.nodeBox.p, sc.flags.p, nodesOut); ++g_kernelLaunches;
  return nLeaves - 1;
}

}  // namespace drt
