// Host-side ownership of device resources: the CUDA error check, the grow-only device buffer and the CUDA event every module uses.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdexcept>
#include <string>
#include <utility>

namespace drt {

#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) throw std::runtime_error(std::string("CUDA error: ") + cudaGetErrorString(e_) + " at " #x); } while (0)

// Grow-only device array, freed with its owner.  ensure(n) makes room for at least n elements; growing waits for `st` before it frees the
// old block (work queued on it may still read it) and, with `keep`, copies the old contents first.  Once warm, nothing on the per-frame path
// allocates: cudaMalloc / cudaFree cost tens to hundreds of ms when they hit the driver's slow path.
template <class T> struct DBuf {
  T* p = nullptr; size_t cap = 0;
  DBuf() = default;
  DBuf(DBuf&& o) noexcept : p(o.p), cap(o.cap) { o.p = nullptr; o.cap = 0; }
  DBuf& operator=(DBuf&& o) noexcept { std::swap(p, o.p); std::swap(cap, o.cap); return *this; }
  ~DBuf() { if (p) cudaFree(p); }
  T* ensure(size_t n, cudaStream_t st, bool keep = false) {
    if (n <= cap) return p;
    size_t nc = n + n / 4 + 1024; T* q = nullptr; CK(cudaMalloc(&q, nc * sizeof(T)));
    if (keep && p && cap) CK(cudaMemcpyAsync(q, p, cap * sizeof(T), cudaMemcpyDeviceToDevice, st));
    if (p) { CK(cudaStreamSynchronize(st)); CK(cudaFree(p)); }
    p = q; cap = nc; return p;
  }
};

// CUDA event created with its owner and destroyed with it
struct DEvent {
  cudaEvent_t e = nullptr;
  DEvent() { CK(cudaEventCreate(&e)); }
  DEvent(DEvent&& o) noexcept : e(o.e) { o.e = nullptr; }
  ~DEvent() { if (e) cudaEventDestroy(e); }
  operator cudaEvent_t() const { return e; }
};

}  // namespace drt
