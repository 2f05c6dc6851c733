// same_owned.h — owned CUDA resources: released when their owner goes, on the device that is current then.
#pragma once

#include <cuda_runtime.h>

#include <utility>

// An array of T from Alloc, released with Free.  grow() allocates before it releases: a failed allocation leaves the
// old array in place and clears the runtime's last error, so that the next launcher does not report it as its own.
template <class T, cudaError_t (*Alloc)(void**, size_t), cudaError_t (*Free)(void*)>
class Buf {
 public:
  Buf() = default;
  Buf(const Buf&) = delete;
  Buf& operator=(const Buf&) = delete;
  ~Buf() { if (p_) Free(p_); }
  operator T*() const { return p_; }
  size_t size() const { return n_; }   // elements
  // room for at least n elements (when it has to grow: n + slack); the contents are not kept
  cudaError_t grow(size_t n, size_t slack = 0) {
    if (n <= n_) return cudaSuccess;
    void* q = nullptr;
    const cudaError_t err = Alloc(&q, (n + slack) * sizeof(T));
    if (err != cudaSuccess) { cudaGetLastError(); return err; }
    if (p_) Free(p_);
    p_ = static_cast<T*>(q); n_ = n + slack;
    return cudaSuccess;
  }
  void swap(Buf& o) { std::swap(p_, o.p_); std::swap(n_, o.n_); }

 private:
  T* p_ = nullptr;
  size_t n_ = 0;
};
template <class T> using DevBuf = Buf<T, cudaMalloc, cudaFree>;
template <class T> using PinnedBuf = Buf<T, cudaMallocHost, cudaFreeHost>;

class Event {
 public:
  Event() = default;
  Event(const Event&) = delete;
  Event& operator=(const Event&) = delete;
  ~Event() { if (ev_) cudaEventDestroy(ev_); }
  cudaError_t create(unsigned flags = cudaEventDefault) { return cudaEventCreateWithFlags(&ev_, flags); }
  operator cudaEvent_t() const { return ev_; }

 private:
  cudaEvent_t ev_ = nullptr;
};

class Stream {
 public:
  Stream() = default;
  Stream(const Stream&) = delete;
  Stream& operator=(const Stream&) = delete;
  ~Stream() { if (st_) cudaStreamDestroy(st_); }
  cudaError_t create() { return cudaStreamCreateWithFlags(&st_, cudaStreamNonBlocking); }
  operator cudaStream_t() const { return st_; }

 private:
  cudaStream_t st_ = nullptr;
};
