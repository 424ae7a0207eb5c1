// dev_buf.h — owner of one cudaMalloc allocation (internal to libdrloco_b200).
//
// Move-only.  The destructor frees the allocation on the device that is current then: the owners of an env's buffers
// are destroyed under that env's DeviceGuard.  alloc / zeros / from_host return the CUDA error of the first call that
// fails; they are meant for buffers built in a local, which is dropped on failure and moved into place on success.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>

#include <utility>
#include <vector>

namespace drl {

template <typename T>
class DevBuf {
 public:
  DevBuf() = default;
  DevBuf(DevBuf&& o) noexcept { swap(o); }
  // the allocation held before goes to o, which frees it
  DevBuf& operator=(DevBuf&& o) noexcept { swap(o); return *this; }
  ~DevBuf() {
    if (p_) cudaFree(p_);
  }
  T* get() const { return p_; }
  size_t size() const { return n_; }

  cudaError_t alloc(size_t n) {             // n elements, uninitialised
    DevBuf b;
    const cudaError_t err = cudaMalloc(&b.p_, n * sizeof(T));
    if (err == cudaSuccess) { b.n_ = n; swap(b); }
    return err;
  }
  cudaError_t zeros(size_t n) {             // n elements, every byte zero
    const cudaError_t err = alloc(n);
    return err != cudaSuccess ? err : cudaMemset(p_, 0, n * sizeof(T));
  }
  template <typename S>
  cudaError_t from_host(const S* src, size_t n) {   // src[0, n), each element converted to T (e.g. double -> float)
    const std::vector<T> tmp(src, src + n);
    const cudaError_t err = alloc(n);
    return err != cudaSuccess ? err : cudaMemcpy(p_, tmp.data(), n * sizeof(T), cudaMemcpyHostToDevice);
  }

 private:
  void swap(DevBuf& o) noexcept { std::swap(p_, o.p_); std::swap(n_, o.n_); }
  T* p_ = nullptr;
  size_t n_ = 0;
};

}  // namespace drl
