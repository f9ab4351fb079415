// Device build of the REFERENCE-topology median-split tree's object order (the parity modes' tree, not the LBVH of lbvh.cuh).
//
// Replaces the per-node TreeMap re-sorting of myBVH.addObjList / buildSortedObjAras (myGeomBase.java:338-386) and the split-axis rule of
// DistRayTracer.getIDXofMaxBVHSpan (DistRayTracer.java:409-418); the host twin is HostScene::refOrderHost (host_scene.cpp), which states why the
// order is a function of the centroid keys alone.  The tree's SHAPE depends only on the object count (split = (int)(.5 * count), leaf at <= 5),
// so the host lays out every level's segments up front and the device does the O(N log^2 N) part level by level:
//   once      per axis: stable radix sort of the 64-bit order-preserving image of the key (two 32-bit rounds) -> dense rank of every object
//             (equal keys share a rank: TreeMap groups them and keeps their arrival order) + the key value of every rank
//   per level per segment: min / max rank per axis (warp-reduced atomics) -> span = key[max] - key[min] in FP64 exactly as the reference forms
//             it -> split axis = first axis of strictly largest span; leaves take axis 0 (a leaf keeps the x-sorted list);
//             then ONE segmented stable sort of the whole array by (segment, rank on the segment's axis): a composite 32-bit key while the
//             bits fit, else a sort by rank followed by a stable sort by segment.  Finished leaves and the object the reference drops at the
//             root (SURVEY Q2) sit in inactive runs whose elements all carry key 0, so the stable sort leaves them in place.
// All sorts are the LSD radix sort of dev_sort.cuh (HBM-bound: per pass 3 x 4 B read + 2 x 4 B written per object).
// Result: the same ord[] array as the host recursion, bit for bit (tests/test_gpu_refbvh.py compares the BVH dumps).
#pragma once
#include "dbuf.h"
#include "dev_sort.cuh"
#include <algorithm>
#include <vector>

namespace drt {

__device__ __forceinline__ unsigned long long rbOrderable(double d) { const unsigned long long b = (unsigned long long)__double_as_longlong(d); return (b >> 63) ? ~b : (b | 0x8000000000000000ull); }

__global__ void k_rb_lowkeys(const double* __restrict__ key, int n, uint32_t* __restrict__ lo) { const int i = blockIdx.x * blockDim.x + threadIdx.x; if (i < n) lo[i] = (uint32_t)rbOrderable(key[i]); }
__global__ void k_rb_highkeys(const double* __restrict__ key, const uint32_t* __restrict__ order, int n, uint32_t* __restrict__ hi) { const int i = blockIdx.x * blockDim.x + threadIdx.x; if (i < n) hi[i] = (uint32_t)(rbOrderable(key[order[i]]) >> 32); }
__global__ void k_rb_flags(const double* __restrict__ key, const uint32_t* __restrict__ order, int n, uint32_t* __restrict__ flag) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x; if (i >= n) return;
  flag[i] = (i > 0 && rbOrderable(key[order[i]]) != rbOrderable(key[order[i - 1]])) ? 1u : 0u;
}
__global__ void k_rb_ranks(const double* __restrict__ key, const uint32_t* __restrict__ order, const uint32_t* __restrict__ exFlag, const uint32_t* __restrict__ flag, int n, uint32_t* __restrict__ rankOfObj, double* __restrict__ keyOfRank) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x; if (i >= n) return;
  const uint32_t r = exFlag[i] + flag[i]; rankOfObj[order[i]] = r; if (flag[i] || i == 0) keyOfRank[r] = key[order[i]];
}
__global__ void k_rb_iota(int n, uint32_t* __restrict__ v) { const int i = blockIdx.x * blockDim.x + threadIdx.x; if (i < n) v[i] = (uint32_t)i; }

// run of position `pos` of this level: last run whose start <= pos
__global__ void k_rb_assign(const int32_t* __restrict__ runStart, int nRuns, int n, uint32_t* __restrict__ runOfPos) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x; if (i >= n) return;
  int lo = 0, hi = nRuns - 1;
  while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (runStart[mid] <= i) lo = mid; else hi = mid - 1; }
  runOfPos[i] = (uint32_t)lo;
}
__global__ void k_rb_init_minmax(int nRuns, uint32_t* __restrict__ mn, uint32_t* __restrict__ mx) { const int i = blockIdx.x * blockDim.x + threadIdx.x; if (i < 3 * nRuns) { mn[i] = 0xFFFFFFFFu; mx[i] = 0u; } }
// kind: 0 inactive, 1 inner node (axis from the spans), 2 leaf (axis 0)
__global__ void k_rb_minmax(const uint32_t* __restrict__ ord, const uint32_t* __restrict__ runOfPos, const int32_t* __restrict__ runKind, const uint32_t* __restrict__ rank0, const uint32_t* __restrict__ rank1, const uint32_t* __restrict__ rank2,
                            int n, int nRuns, uint32_t* __restrict__ mn, uint32_t* __restrict__ mx) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x; const bool ok = i < n;
  const uint32_t run = ok ? runOfPos[i] : 0xFFFFFFFFu; const bool act = ok && runKind[run] == 1;
  uint32_t r[3] = {0, 0, 0}; if (act) { const uint32_t o = ord[i]; r[0] = rank0[o]; r[1] = rank1[o]; r[2] = rank2[o]; }
  const uint32_t run0 = __shfl_sync(0xffffffffu, run, 0);
  if (__all_sync(0xffffffffu, run == run0)) {           // the usual case near the root: the whole warp sits in one segment
    if (!__any_sync(0xffffffffu, act)) return;
#pragma unroll
    for (int a = 0; a < 3; ++a) { const uint32_t lo = __reduce_min_sync(0xffffffffu, r[a]), hi = __reduce_max_sync(0xffffffffu, r[a]);
      if ((threadIdx.x & 31) == 0) { atomicMin(&mn[a * nRuns + run0], lo); atomicMax(&mx[a * nRuns + run0], hi); } }
  } else if (act) {
#pragma unroll
    for (int a = 0; a < 3; ++a) { atomicMin(&mn[a * nRuns + run], r[a]); atomicMax(&mx[a * nRuns + run], r[a]); }
  }
}
// DistRayTracer.getIDXofMaxBVHSpan: diff = last - first of the list sorted on coordinate i; `if (maxSpan < diff)` from maxSpan = -1, i = 0, 1, 2
__global__ void k_rb_axis(int nRuns, const int32_t* __restrict__ runKind, const uint32_t* __restrict__ mn, const uint32_t* __restrict__ mx, const double* __restrict__ key0, const double* __restrict__ key1, const double* __restrict__ key2,
                          int32_t* __restrict__ axisOut, unsigned int* __restrict__ err) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x; if (r >= nRuns) return;
  const int kind = runKind[r]; int axis = 3;
  if (kind == 2) axis = 0;
  else if (kind == 1) {
    const double* keyOfRank[3] = {key0, key1, key2}; double widest = -1; axis = -1;
    for (int a = 0; a < 3; ++a) { const double span = keyOfRank[a][mx[a * nRuns + r]] - keyOfRank[a][mn[a * nRuns + r]]; if (widest < span) { widest = span; axis = a; } }
    if (axis < 0) { atomicOr(err, 1u); axis = 3; }
  }
  axisOut[r] = axis;
}
// sort key of every position: rank of its object on its run's axis (0 in inactive runs); composite: the run index sits above the rank bits
__global__ void k_rb_keys(const uint32_t* __restrict__ ord, const uint32_t* __restrict__ runOfPos, const int32_t* __restrict__ axisOfRun, const uint32_t* __restrict__ rank0, const uint32_t* __restrict__ rank1, const uint32_t* __restrict__ rank2,
                          int n, int rankBits, int composite, uint32_t* __restrict__ keyOut) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x; if (i >= n) return;
  const uint32_t run = runOfPos[i]; const int ax = axisOfRun[run]; const uint32_t o = ord[i];
  const uint32_t r = ax == 0 ? rank0[o] : ax == 1 ? rank1[o] : ax == 2 ? rank2[o] : 0u;
  keyOut[i] = composite ? ((run << rankBits) | r) : r;
}
__global__ void k_rb_gather(const uint32_t* __restrict__ src, const uint32_t* __restrict__ idx, int n, uint32_t* __restrict__ dst) { const int i = blockIdx.x * blockDim.x + threadIdx.x; if (i < n) dst[i] = src[idx[i]]; }

struct RefBvhScratch {
  DBuf<double> key[3], keyOfRank[3]; DBuf<uint32_t> rank[3], keys[2], vals[2], ord[2], runOfPos, flag, hist, sortScan, rankScan, mn, mx;
  DBuf<int32_t> runStart, runKind, axis; DBuf<unsigned int> err; DEvent ev[2];
  void ensure(size_t n, size_t runs, cudaStream_t st) {
    for (int a = 0; a < 3; ++a) { key[a].ensure(n, st); keyOfRank[a].ensure(n, st); rank[a].ensure(n, st); }
    for (int k = 0; k < 2; ++k) { keys[k].ensure(n, st); vals[k].ensure(n, st); ord[k].ensure(n, st); }
    runOfPos.ensure(n, st); flag.ensure(n, st);
    const long long nb = radixBlocks((long long)n);
    hist.ensure((size_t)256 * nb, st); sortScan.ensure((size_t)scanScratchWords(256 * nb), st); rankScan.ensure((size_t)scanScratchWords((long long)n), st); err.ensure(1, st);
    runStart.ensure(runs, st); runKind.ensure(runs, st); axis.ensure(runs, st); mn.ensure(3 * runs, st); mx.ensure(3 * runs, st);
  }
};

// keysHost = [3][n]; ordHost[n] receives the order.  Returns false when the device cannot decide (NaN / infinite spans): the host recursion then
// reports the error exactly as before.  msOut: CUDA-event time of everything between the H2D of the keys and the D2H of the order.
static inline bool refOrderDevice(int n, const double* keysHost, int32_t* ordHost, RefBvhScratch& sc, cudaStream_t st, double* msOut) {
  if (n < 2) return false;
  for (size_t i = 0; i < (size_t)3 * n; ++i) if (keysHost[i] != keysHost[i]) return false;
  // ---- every level's runs, from the count alone
  struct Seg { int s, m, count; };
  std::vector<int32_t> runStart, runKind; std::vector<int> lvlOff, lvlRuns;
  { std::vector<Seg> cur{{0, n, n - 1}}, next;
    while (!cur.empty()) {
      lvlOff.push_back((int)runStart.size()); int pos = 0;
      for (const Seg& g : cur) { if (g.s > pos) { runStart.push_back(pos); runKind.push_back(0); } runStart.push_back(g.s); runKind.push_back(g.count <= 5 ? 2 : 1); pos = g.s + g.m; }
      if (pos < n) { runStart.push_back(pos); runKind.push_back(0); }
      lvlRuns.push_back((int)runStart.size() - lvlOff.back());
      next.clear();
      for (const Seg& g : cur) if (g.count > 5) { const int split = (int)(.5 * g.count); next.push_back({g.s, split, split}); next.push_back({g.s + split, g.count - split, g.count - split}); }
      cur.swap(next);
    } }
  sc.ensure((size_t)n, runStart.size(), st);
  CK(cudaEventRecord(sc.ev[0], st));
  for (int a = 0; a < 3; ++a) CK(cudaMemcpyAsync(sc.key[a].p, keysHost + (size_t)a * n, (size_t)n * 8, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(sc.runStart.p, runStart.data(), runStart.size() * 4, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(sc.runKind.p, runKind.data(), runKind.size() * 4, cudaMemcpyHostToDevice, st));
  CK(cudaMemsetAsync(sc.err.p, 0, 4, st));
  const unsigned gN = (unsigned)((n + 255) / 256);
  int rankBits = 1; while ((1ll << rankBits) < (long long)n) ++rankBits;
  uint32_t* keys[2] = {sc.keys[0].p, sc.keys[1].p}; uint32_t* vals[2] = {sc.vals[0].p, sc.vals[1].p};
  const uint32_t* rank[3] = {sc.rank[0].p, sc.rank[1].p, sc.rank[2].p}; const double* keyOfRank[3] = {sc.keyOfRank[0].p, sc.keyOfRank[1].p, sc.keyOfRank[2].p};
  uint32_t* ord[2] = {sc.ord[0].p, sc.ord[1].p};
  // ---- dense ranks per axis
  for (int a = 0; a < 3; ++a) {
    k_rb_lowkeys<<<gN, 256, 0, st>>>(sc.key[a].p, n, keys[0]); ++g_kernelLaunches;
    int cur = radixSortPairs(keys, vals, n, 32, true, sc.hist.p, sc.sortScan.p, st);
    uint32_t* k2[2] = {keys[cur ^ 1], keys[cur]}; uint32_t* v2[2] = {vals[cur], vals[cur ^ 1]};
    k_rb_highkeys<<<gN, 256, 0, st>>>(sc.key[a].p, v2[0], n, k2[0]); ++g_kernelLaunches;
    const int c2 = radixSortPairs(k2, v2, n, 32, false, sc.hist.p, sc.sortScan.p, st);
    const uint32_t* order = v2[c2];
    k_rb_flags<<<gN, 256, 0, st>>>(sc.key[a].p, order, n, sc.flag.p); ++g_kernelLaunches;
    scanExclusiveU32(sc.flag.p, sc.runOfPos.p, n, sc.rankScan.p, st);
    k_rb_ranks<<<gN, 256, 0, st>>>(sc.key[a].p, order, sc.runOfPos.p, sc.flag.p, n, sc.rank[a].p, sc.keyOfRank[a].p); ++g_kernelLaunches;
  }
  // ---- levels
  int oc = 0; k_rb_iota<<<gN, 256, 0, st>>>(n, ord[0]); ++g_kernelLaunches;
  for (size_t L = 0; L < lvlOff.size(); ++L) {
    const int nRuns = lvlRuns[L]; const int32_t* rs = sc.runStart.p + lvlOff[L]; const int32_t* rk = sc.runKind.p + lvlOff[L]; int32_t* ax = sc.axis.p + lvlOff[L];
    const unsigned gR = (unsigned)((3 * nRuns + 255) / 256);
    k_rb_assign<<<gN, 256, 0, st>>>(rs, nRuns, n, sc.runOfPos.p);
    k_rb_init_minmax<<<gR, 256, 0, st>>>(nRuns, sc.mn.p, sc.mx.p);
    k_rb_minmax<<<gN, 256, 0, st>>>(ord[oc], sc.runOfPos.p, rk, rank[0], rank[1], rank[2], n, nRuns, sc.mn.p, sc.mx.p);
    k_rb_axis<<<(unsigned)((nRuns + 255) / 256), 256, 0, st>>>(nRuns, rk, sc.mn.p, sc.mx.p, keyOfRank[0], keyOfRank[1], keyOfRank[2], ax, sc.err.p);
    int runBits = 1; while ((1ll << runBits) < (long long)nRuns) ++runBits;
    const int composite = (runBits + rankBits <= 32) ? 1 : 0;
    k_rb_keys<<<gN, 256, 0, st>>>(ord[oc], sc.runOfPos.p, ax, rank[0], rank[1], rank[2], n, rankBits, composite, keys[0]);
    g_kernelLaunches += 5;
    const uint32_t* perm;
    if (composite) { const int c = radixSortPairs(keys, vals, n, nRuns > 1 ? runBits + rankBits : rankBits, true, sc.hist.p, sc.sortScan.p, st); perm = vals[c]; }
    else {
      const int c = radixSortPairs(keys, vals, n, rankBits, true, sc.hist.p, sc.sortScan.p, st);
      uint32_t* k2[2] = {keys[c ^ 1], keys[c]}; uint32_t* v2[2] = {vals[c], vals[c ^ 1]};
      k_rb_gather<<<gN, 256, 0, st>>>(sc.runOfPos.p, v2[0], n, k2[0]); ++g_kernelLaunches;
      const int c2 = radixSortPairs(k2, v2, n, runBits, false, sc.hist.p, sc.sortScan.p, st); perm = v2[c2];
    }
    k_rb_gather<<<gN, 256, 0, st>>>(ord[oc], perm, n, ord[oc ^ 1]); ++g_kernelLaunches; oc ^= 1;
  }
  unsigned int err = 0;
  CK(cudaMemcpyAsync(ordHost, ord[oc], (size_t)n * 4, cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(&err, sc.err.p, 4, cudaMemcpyDeviceToHost, st));
  CK(cudaEventRecord(sc.ev[1], st)); CK(cudaStreamSynchronize(st));
  float ms = 0; CK(cudaEventElapsedTime(&ms, sc.ev[0], sc.ev[1])); if (msOut) *msOut = ms;
  return err == 0;
}

}  // namespace drt
