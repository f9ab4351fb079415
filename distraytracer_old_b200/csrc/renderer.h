// Host-side handle of the wavefront renderer (device memory owner + kernel launcher).
#pragma once
#include "host_scene.h"
#include <memory>
#include <string>
#include <vector>

namespace drt {

struct RenderStats {
  unsigned long long primary, shadow, reflect, refract, photonSeg;   // logical rays (SURVEY Q13)
  unsigned long long boxTests, primTests, boxTestsClosest, primTestsClosest;   // only when counters are enabled
  unsigned long long photonsStored;
  unsigned long long kernelLaunches;
  unsigned long long deferred, retries, hostSyncs;                    // rays / light records the lean kernels left to the generic pass; re-rendered frames; host syncs of the call
  double msTrace, msShade, msLight, msOther, msTotal;               // CUDA-event times of the last render call
};

struct RenderOutputs {           // device pointers, any may be null; sized cols*rows (rgb: 3x)
  int32_t* argb; int32_t* hitPrim; int32_t* hitInst; double* rgb; double* t;
  int32_t packed;                // != 0: argb is indexed by the rank's COMPACT pixel index (its chunks back to back) instead of the absolute pixel
};

class Renderer {
 public:
  Renderer(int device);
  ~Renderer();
  void upload(const HostScene& hs, bool sameScene = false);   // flat scene -> HBM (sameScene: a re-upload of what is already resident, keeps the depth hint)
  bool orderBvh(int n, const double* keys3n, int32_t* ord, double* msDevice);   // device twin of HostScene::refOrderHost (csrc/refbvh.cuh)
  void setBatchRays(long long n) { batchRays_ = n; }
  void setCounters(bool on) { counters_ = on; }
  void setAccelMode(int m) { accelMode_ = m; }              // DRT_ACCEL_*: takes effect at the next upload
  // render pixels [pix0, pix1) (row-major pixel indices) into the device buffers of `out` (indexed by absolute pixel)
  void renderRange(long long pix0, long long pix1, const RenderOutputs& out, RenderStats* stats);
  void renderChunks(long long pix0, long long pix1, int world, int rank, int chunkRows, const RenderOutputs& out, RenderStats* stats);
  // full frame to host memory (D2H inside)
  void renderToHost(int32_t* argbHost, int32_t* hitPrimHost, int32_t* hitInstHost, double* rgbHost, double* tHost, RenderStats* stats);
  // explicit world-space rays (closest hit only) for parity tests: ids = {primSerial, instSerial} per ray
  void traceRays(long long n, const double* orgHost, const double* dirHost, int32_t* idsHost, double* tHost);
  // caller rays in DEVICE memory (include/drt.h drt_query_closest / drt_query_occluded); every pointer is a device pointer, optional ones may
  // be null (tmax: +inf; pos, nrm: not written).  Complete when the call returns; stats: launches, deferred rays, one host sync, event ms
  void queryClosest(long long n, const double* org, const double* dir, const double* tmax, int32_t* ids, double* t, double* pos, double* nrm, RenderStats* stats);
  void queryOccluded(long long n, const double* org, const double* dir, const double* dist, uint8_t* occluded, RenderStats* stats);
  void evalTexture(int shaderIdx, long long n, const double* hitLocHost, const double* fwdLocHost, double* outHost);
  void emitPhotons(RenderStats* stats);               // builds the photon map if the scene asks for one
  long long getPhotons(double* out6Host, long long cap);
  void emitPhotonsRange(long long i0, long long i1, RenderStats* stats);          // photon indices [i0,i1) of every light, no grid build
  long long exportPhotonsDevice(double* dst6Dev, long long cap);                  // canonical-order records -> caller's device buffer; returns count
  void buildPhotonsFromDevice(const double* src6Dev, long long n, RenderStats* stats);   // replace the record set (e.g. all-gathered) and build the grid
  void probePhotons(long long n, const double* ptsHost, double* out5Host);       // per point: sum r,g,b of the k nearest, d^2 of the farthest, candidates visited
  // ---- multi-GPU inside the library: one Renderer per rank, NCCL (loaded at run time) on the renderer's own stream
  static void commUniqueId(unsigned char id128[128]);
  void commInit(const unsigned char id128[128], int world, int rank);
  void commDestroy();
  int commWorld() const { return world_; }
  int commRank() const { return rank_; }
  // this rank's interleaved row chunks -> NCCL send/recv gather -> assembled frame on rank 0 (device and/or host buffer; both may be null on
  // other ranks).  Photon scenes: emission split by photon index, records all-gathered, grid built on every rank.
  // the partition itself (pure host functions, also behind the C ABI so that the world-size-2 CPU tests exercise the shipped mapping)
  static long long distRankPixels(int cols, int rows, int world, int rank, int chunkRows);                 // compact pixels rank `rank` renders (whole chunks)
  static long long distAbsPixel(int cols, int rows, int world, int rank, int chunkRows, long long compact);   // absolute pixel of a compact slot, -1 beyond the frame
  static void distPhotonRange(long long nCast, int world, int rank, long long out2[2]);
  void renderDistributed(int32_t* argbHostRank0, int32_t* argbDevRank0, int chunkRows, bool reemitPhotons, RenderStats* stats);
  long long probeFastBvh(int fastIndex, std::vector<FTri>& tris, std::vector<FNode>& nodes, int32_t info[4]);   // resident packed triangles (+ LBVH nodes) of a fast BVH
  void accelInfo(double out[4]) const;                 // LBVH build ms (CUDA events), triangles and nodes it covers, scene bytes in HBM
  int cols() const { return g_.cols; }
  int rows() const { return g_.rows; }
  int spp() const { return g_.spp; }
  void* stream() const { return stream_; }
  const FGlobals& globals() const { return g_; }
  struct Impl;

 private:
  std::unique_ptr<Impl> impl_;
  FGlobals g_;
  int device_;
  void* stream_;
  long long batchRays_ = 8ll << 20;
  bool counters_ = false;
  int accelMode_ = 0;
  bool keepDepthHint_ = false;
  void* comm_ = nullptr; int world_ = 1, rank_ = 0;
};

}  // namespace drt
