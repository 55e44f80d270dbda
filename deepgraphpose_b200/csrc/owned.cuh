// Owner types of every CUDA resource the library holds: device and pinned host memory, events, streams, graphs and graph
// executables.  An owning member is one of these types; a raw pointer or handle is only ever a view into one of them, so
// destroying the owner (ultimately `delete h` in dgp_destroy, after a device synchronize) releases everything, and every
// early return of an error path releases what was allocated before it.
//
// Destructors ignore errors: they run during teardown and unwinding, where there is nobody to report to.  Owners are never
// static or global: a destructor that runs at process exit would run after the CUDA runtime has been torn down.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include <atomic>
#include <memory>

namespace dgp {

// Process-wide count of live owned resources (dgp_debug_live_resources): objects of every kind, bytes of device memory.
extern std::atomic<int64_t> g_live_objects, g_live_device_bytes;

// Device (Pinned = false, cudaMalloc) or pinned host (Pinned = true, cudaHostAlloc) memory.
template <bool Pinned>
class Mem {
 public:
  Mem() = default;
  Mem(Mem&& o) noexcept : p_(o.p_), bytes_(o.bytes_) { o.p_ = nullptr; o.bytes_ = 0; }
  Mem& operator=(Mem&& o) noexcept {
    if (this != &o) {
      reset();
      p_ = o.p_; bytes_ = o.bytes_;
      o.p_ = nullptr; o.bytes_ = 0;
    }
    return *this;
  }
  Mem(const Mem&) = delete;
  Mem& operator=(const Mem&) = delete;
  ~Mem() { reset(); }

  // Releases what is held, then allocates `bytes`; on failure the owner holds nothing.
  cudaError_t alloc(size_t bytes) {
    reset();
    void* p = nullptr;
    const cudaError_t e = Pinned ? cudaHostAlloc(&p, bytes, cudaHostAllocDefault) : cudaMalloc(&p, bytes);
    if (e != cudaSuccess) return e;
    p_ = p;
    bytes_ = bytes;
    ++g_live_objects;
    if (!Pinned) g_live_device_bytes += (int64_t)bytes;
    return cudaSuccess;
  }
  void reset() {
    if (!p_) return;
    if (Pinned) cudaFreeHost(p_);
    else cudaFree(p_);
    --g_live_objects;
    if (!Pinned) g_live_device_bytes -= (int64_t)bytes_;
    p_ = nullptr;
    bytes_ = 0;
  }
  void* get() const { return p_; }
  template <class T>
  T* get() const { return static_cast<T*>(p_); }
  size_t bytes() const { return bytes_; }

 private:
  void* p_ = nullptr;
  size_t bytes_ = 0;
};
using DevBuf = Mem<false>;
using PinnedBuf = Mem<true>;

template <class T, cudaError_t (*Destroy)(T*)>
struct CudaDeleter {
  void operator()(T* p) const {
    Destroy(p);
    --g_live_objects;
  }
};
using Event = std::unique_ptr<CUevent_st, CudaDeleter<CUevent_st, cudaEventDestroy>>;
using Stream = std::unique_ptr<CUstream_st, CudaDeleter<CUstream_st, cudaStreamDestroy>>;
using Graph = std::unique_ptr<CUgraph_st, CudaDeleter<CUgraph_st, cudaGraphDestroy>>;
using GraphExec = std::unique_ptr<CUgraphExec_st, CudaDeleter<CUgraphExec_st, cudaGraphExecDestroy>>;

// Hands a freshly created object to its owner (which releases whatever it held before).
template <class Owner>
void adopt(Owner* o, typename Owner::pointer p) {
  o->reset(p);
  ++g_live_objects;
}

inline cudaError_t create(Event* e, unsigned flags) {
  cudaEvent_t p = nullptr;
  const cudaError_t r = cudaEventCreateWithFlags(&p, flags);
  if (r == cudaSuccess) adopt(e, p);
  return r;
}
inline cudaError_t create(Stream* s, unsigned flags) {
  cudaStream_t p = nullptr;
  const cudaError_t r = cudaStreamCreateWithFlags(&p, flags);
  if (r == cudaSuccess) adopt(s, p);
  return r;
}

}  // namespace dgp
