// Device-wide primitives shared by the photon hash-grid build and the LBVH builder: exclusive scan (u32) and a stable
// LSD radix sort of (u32 key, u32 value) pairs, 8 bits per pass.  Hand-written for sm_100a; HBM-bound (each pass reads the
// keys twice and the values once, writes both once), no library sort on the product path.
//
// These replace the reference's object-level sorting: myKD_Tree.build_tree's Collections.sort per level
// (myLight.java:325-381) and myBVH.buildSortedObjAras' TreeMap re-sorting per node (myGeomBase.java:338-357).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdexcept>

namespace drt {

static thread_local unsigned long long g_kernelLaunches = 0;   // every launch of the build-side kernels (sort, scan, photon map, LBVH) bumps this; the renderer folds it into its stats

// ---------------------------------------------------------------------------------------------------------------
// exclusive scan, u32, any n: 256 threads x 8 items per block, block sums scanned recursively
// ---------------------------------------------------------------------------------------------------------------
#define DRT_SCAN_ITEMS 8
#define DRT_SCAN_TILE (256 * DRT_SCAN_ITEMS)

__device__ __forceinline__ uint32_t blockExclusiveScan256(uint32_t v, uint32_t* warpSums /*[8] shared*/, uint32_t& blockTotal) {
  const unsigned lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  uint32_t incl = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { uint32_t t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= (unsigned)o) incl += t; }
  if (lane == 31) warpSums[w] = incl;
  __syncthreads();
  uint32_t base = 0, tot = 0;
#pragma unroll
  for (int i = 0; i < 8; ++i) { uint32_t s = warpSums[i]; if (i < (int)w) base += s; tot += s; }
  blockTotal = tot;
  __syncthreads();
  return base + incl - v;
}

// pass 1: per-tile totals
__global__ void __launch_bounds__(256) k_scan_tile_sums(const uint32_t* __restrict__ in, long long n, uint32_t* __restrict__ tileSums) {
  __shared__ uint32_t ws[8];
  long long base = (long long)blockIdx.x * DRT_SCAN_TILE + (long long)threadIdx.x * DRT_SCAN_ITEMS; uint32_t s = 0;
#pragma unroll
  for (int i = 0; i < DRT_SCAN_ITEMS; ++i) if (base + i < n) s += in[base + i];
  uint32_t tot; blockExclusiveScan256(s, ws, tot);
  if (threadIdx.x == 0) tileSums[blockIdx.x] = tot;
}
// pass 3: rescan each tile with its scanned base
__global__ void __launch_bounds__(256) k_scan_apply(const uint32_t* __restrict__ in, long long n, const uint32_t* __restrict__ tileBase, uint32_t* __restrict__ out) {
  __shared__ uint32_t ws[8];
  long long base = (long long)blockIdx.x * DRT_SCAN_TILE + (long long)threadIdx.x * DRT_SCAN_ITEMS; uint32_t v[DRT_SCAN_ITEMS], s = 0;
#pragma unroll
  for (int i = 0; i < DRT_SCAN_ITEMS; ++i) { v[i] = (base + i < n) ? in[base + i] : 0u; s += v[i]; }
  uint32_t tot; uint32_t ex = blockExclusiveScan256(s, ws, tot) + (tileBase ? tileBase[blockIdx.x] : 0u);
#pragma unroll
  for (int i = 0; i < DRT_SCAN_ITEMS; ++i) { if (base + i < n) out[base + i] = ex; ex += v[i]; }
}

// scratch must hold scanScratchWords(n) u32. in may alias out.
static inline long long scanScratchWords(long long n) { long long w = 0; while (n > 1) { n = (n + DRT_SCAN_TILE - 1) / DRT_SCAN_TILE; w += n + 1; if (n == 1) break; } return w + 2; }
static inline void scanExclusiveU32(const uint32_t* in, uint32_t* out, long long n, uint32_t* scratch, cudaStream_t st) {
  if (n <= 0) return;
  long long tiles = (n + DRT_SCAN_TILE - 1) / DRT_SCAN_TILE;
  if (tiles == 1) { k_scan_apply<<<1, 256, 0, st>>>(in, n, nullptr, out); ++g_kernelLaunches; return; }
  uint32_t* sums = scratch;
  k_scan_tile_sums<<<(unsigned)tiles, 256, 0, st>>>(in, n, sums); ++g_kernelLaunches;
  scanExclusiveU32(sums, sums, tiles, scratch + tiles + 1, st);
  k_scan_apply<<<(unsigned)tiles, 256, 0, st>>>(in, n, sums, out); ++g_kernelLaunches;
}

// ---------------------------------------------------------------------------------------------------------------
// stable LSD radix sort of (key, value) pairs
// ---------------------------------------------------------------------------------------------------------------
#define DRT_RS_ITEMS 16                      // keys per thread
#define DRT_RS_TILE (256 * DRT_RS_ITEMS)     // keys per block; warp w owns the contiguous slice [w*512, w*512+512) of the tile

// per-warp digit counts of this block's tile -> cnt[w][d]; every key is visited in index order by its warp
__device__ __forceinline__ void rsCountWarp(const uint32_t* __restrict__ keys, long long n, long long warpBase, int shift, uint32_t* cntW /*[256] shared, this warp*/, uint32_t kreg[DRT_RS_ITEMS]) {
  const unsigned lane = threadIdx.x & 31;
#pragma unroll
  for (int r = 0; r < DRT_RS_ITEMS; ++r) {
    long long idx = warpBase + r * 32 + lane; bool ok = idx < n;
    uint32_t k = ok ? keys[idx] : 0xFFFFFFFFu; kreg[r] = k;
    uint32_t d = ok ? ((k >> shift) & 255u) : 256u;
    unsigned peers = __match_any_sync(0xffffffffu, d);
    if (ok && (unsigned)(__ffs(peers) - 1) == lane) cntW[d] += __popc(peers);
    __syncwarp();
  }
}

__global__ void __launch_bounds__(256) k_radix_hist(const uint32_t* __restrict__ keys, long long n, int shift, uint32_t* __restrict__ hist /*[256][numBlocks]*/) {
  __shared__ uint32_t cnt[8][256];
  for (int i = threadIdx.x; i < 8 * 256; i += 256) (&cnt[0][0])[i] = 0;
  __syncthreads();
  const unsigned w = threadIdx.x >> 5; uint32_t kreg[DRT_RS_ITEMS];
  rsCountWarp(keys, n, (long long)blockIdx.x * DRT_RS_TILE + (long long)w * (32 * DRT_RS_ITEMS), shift, cnt[w], kreg);
  __syncthreads();
  uint32_t tot = 0;
#pragma unroll
  for (int i = 0; i < 8; ++i) tot += cnt[i][threadIdx.x];
  hist[(long long)threadIdx.x * gridDim.x + blockIdx.x] = tot;
}

__global__ void __launch_bounds__(256) k_radix_scatter(const uint32_t* __restrict__ keysIn, const uint32_t* __restrict__ valsIn, uint32_t* __restrict__ keysOut, uint32_t* __restrict__ valsOut,
                                                       long long n, int shift, const uint32_t* __restrict__ histScanned) {
  __shared__ uint32_t cnt[8][256];
  for (int i = threadIdx.x; i < 8 * 256; i += 256) (&cnt[0][0])[i] = 0;
  __syncthreads();
  const unsigned w = threadIdx.x >> 5, lane = threadIdx.x & 31; uint32_t kreg[DRT_RS_ITEMS];
  const long long warpBase = (long long)blockIdx.x * DRT_RS_TILE + (long long)w * (32 * DRT_RS_ITEMS);
  rsCountWarp(keysIn, n, warpBase, shift, cnt[w], kreg);
  __syncthreads();
  {   // thread d: turn the per-warp counts of digit d into output offsets (global base + earlier warps of this block)
    uint32_t run = histScanned[(long long)threadIdx.x * gridDim.x + blockIdx.x];
#pragma unroll
    for (int i = 0; i < 8; ++i) { uint32_t c = cnt[i][threadIdx.x]; cnt[i][threadIdx.x] = run; run += c; }
  }
  __syncthreads();
  uint32_t* off = cnt[w];
#pragma unroll
  for (int r = 0; r < DRT_RS_ITEMS; ++r) {
    long long idx = warpBase + r * 32 + lane; bool ok = idx < n;
    uint32_t k = kreg[r]; uint32_t d = ok ? ((k >> shift) & 255u) : 256u;
    unsigned peers = __match_any_sync(0xffffffffu, d);
    uint32_t pos = 0;
    if (ok) pos = off[d] + __popc(peers & ((1u << lane) - 1u));
    __syncwarp();
    if (ok && (unsigned)(__ffs(peers) - 1) == lane) off[d] += __popc(peers);
    __syncwarp();
    if (ok) { keysOut[pos] = k; valsOut[pos] = valsIn ? valsIn[idx] : (uint32_t)idx; }
  }
}

// Sorts n pairs by the low `bits` bits of the key. Buffers: keys[2], vals[2] (ping-pong, each n words); returns the index (0/1) of
// the buffer that holds the result. vals[0] may be nullptr on entry semantics: pass identity=true to generate 0..n-1 in the first pass.
// hist: 256*numBlocks words, scratch: scanScratchWords(256*numBlocks).
static inline long long radixBlocks(long long n) { return (n + DRT_RS_TILE - 1) / DRT_RS_TILE; }
static inline int radixSortPairs(uint32_t* keys[2], uint32_t* vals[2], long long n, int bits, bool identity, uint32_t* hist, uint32_t* scratch, cudaStream_t st) {
  int cur = 0; if (n <= 0) return 0;
  const long long nb = radixBlocks(n);
  for (int shift = 0; shift < bits; shift += 8) {
    k_radix_hist<<<(unsigned)nb, 256, 0, st>>>(keys[cur], n, shift, hist); ++g_kernelLaunches;
    scanExclusiveU32(hist, hist, 256 * nb, scratch, st);
    k_radix_scatter<<<(unsigned)nb, 256, 0, st>>>(keys[cur], (identity && shift == 0) ? nullptr : vals[cur], keys[cur ^ 1], vals[cur ^ 1], n, shift, hist); ++g_kernelLaunches;
    cur ^= 1;
  }
  if (bits <= 0 && identity) throw std::runtime_error("radixSortPairs: bits must be > 0");
  return cur;
}

}  // namespace drt
