// rtrb_devbuf.h — the device array that owns every allocation of a renderer (rtrb_api.cu, rtrb_png.cu).
#ifndef RTRB_DEVBUF_H
#define RTRB_DEVBUF_H

#include <cuda_runtime.h>
#include <stddef.h>

// Grows on demand and is freed with its owner; its device must be current whenever it grows or is destroyed.
// Move-only: moving hands the allocation over without changing its address.
template <typename T>
struct DevBuf {
  T* p = nullptr;
  size_t n = 0;  // capacity in elements

  DevBuf() = default;
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  DevBuf(DevBuf&& o) noexcept : p(o.p), n(o.n) { o.p = nullptr; o.n = 0; }
  ~DevBuf() { release(); }

  // At least `want` elements.  A smaller array is freed first: growing loses the contents.
  cudaError_t ensure(size_t want) {
    if (want <= n && p) return cudaSuccess;
    release();
    if (want == 0) return cudaSuccess;
    cudaError_t e = cudaMalloc((void**)&p, want * sizeof(T));
    if (e == cudaSuccess) n = want;
    return e;
  }

  // Takes over `q` (count elements, from cudaMalloc) in place of the current allocation, which is freed.
  void adopt(T* q, size_t count) {
    release();
    p = q;
    n = count;
  }

  // Hands the allocation over to the caller (who frees it with cudaFree) and leaves the array empty.
  T* detach() {
    T* q = p;
    p = nullptr;
    n = 0;
    return q;
  }

 private:
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    n = 0;
  }
};

#endif  // RTRB_DEVBUF_H
