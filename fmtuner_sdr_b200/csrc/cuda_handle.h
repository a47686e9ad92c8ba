// Owning handles for the CUDA resources of an engine or a channelizer: device memory, streams and
// events. A handle is move-only and releases its resource when it is destroyed while non-null, so an
// object that holds its resources in handles frees all of them when it is deleted, on every path.
// A handle converts implicitly to the raw pointer or handle and is passed wherever that is expected.
// The owner makes the resource's device current before it destroys the handle.
#ifndef FMGPU_CUDA_HANDLE_H_
#define FMGPU_CUDA_HANDLE_H_

#include <cuda_runtime.h>

#include <algorithm>
#include <cstddef>
#include <utility>

namespace fmgpu {

template <typename H, cudaError_t (*Release)(H)>
class CudaHandle {
 public:
  CudaHandle() = default;
  CudaHandle(CudaHandle &&o) noexcept : h_(std::exchange(o.h_, nullptr)) {}  // copying is deleted
  CudaHandle &operator=(CudaHandle &&o) noexcept {
    std::swap(h_, o.h_);  // o releases what this held
    return *this;
  }
  ~CudaHandle() {
    if (h_) {
      Release(h_);
    }
  }

  operator H() const { return h_; }
  H get() const { return h_; }

  // Releases what is held and returns the slot for a cudaMalloc, cudaStreamCreate* or
  // cudaEventCreate* call to fill.
  H *out() {
    *this = CudaHandle();
    return &h_;
  }

 private:
  H h_ = nullptr;
};

template <typename T> cudaError_t freeDevice(T *p) { return cudaFree(p); }

template <typename T> using DeviceArray = CudaHandle<T *, freeDevice<T>>;
using Stream = CudaHandle<cudaStream_t, cudaStreamDestroy>;
using Event = CudaHandle<cudaEvent_t, cudaEventDestroy>;

// count elements of device memory (at least one), zero-filled
template <typename T> cudaError_t devAlloc(DeviceArray<T> *p, size_t count) {
  const size_t bytes = std::max<size_t>(1, count) * sizeof(T);
  cudaError_t err = cudaMalloc(reinterpret_cast<void **>(p->out()), bytes);
  if (err == cudaSuccess) {
    err = cudaMemset(*p, 0, bytes);
  }
  return err;
}

}  // namespace fmgpu

#endif  // FMGPU_CUDA_HANDLE_H_
