// fiesta_b200 -- owners of device (cudaMalloc) and pinned host (cudaMallocHost) memory; host code only.  Every buffer of the
// library is one of these: it is freed by its owner's destructor, so create / destroy functions keep no pointer lists.
// The caller makes the owning device current before an owner is destroyed.  Kernels and CUB still take raw pointers: an
// owner converts to T* implicitly (get() where a template would deduce the owner type itself).
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <utility>

template <typename T, bool PINNED>
class FbBuf {
 public:
  FbBuf() = default;
  FbBuf(const FbBuf &) = delete;
  FbBuf &operator=(const FbBuf &) = delete;
  FbBuf(FbBuf &&o) noexcept { swap(o); }
  FbBuf &operator=(FbBuf &&o) noexcept { FbBuf(std::move(o)).swap(*this); return *this; }
  ~FbBuf() {
    if (p_ && PINNED) cudaFreeHost(p_);
    else if (p_) cudaFree(p_);
  }

  // Exactly n elements, contents undefined; the old block is freed first.
  cudaError_t alloc(size_t n) {
    *this = FbBuf();
    void *p = nullptr;
    const cudaError_t e = PINNED ? cudaMallocHost(&p, n * sizeof(T)) : cudaMalloc(&p, n * sizeof(T));
    if (e == cudaSuccess) { p_ = static_cast<T *>(p); n_ = n; }
    return e;
  }
  // At least `need` elements.  Growth allocates need * 1.5 + 1 MiB, so a slowly growing demand reallocates rarely.  keep:
  // the old contents are copied on stream s and the copy is waited for before the old block is freed.  On an error the
  // buffer is left as it was.
  cudaError_t reserve(size_t need, cudaStream_t s, bool keep) {
    if (need <= n_) return cudaSuccess;
    FbBuf b;
    cudaError_t e = b.alloc(need + need / 2 + (size_t(1) << 20) / sizeof(T));
    if (e == cudaSuccess && keep && n_) e = cudaMemcpyAsync(b.p_, p_, n_ * sizeof(T), cudaMemcpyDefault, s);
    if (e == cudaSuccess && keep && n_) e = cudaStreamSynchronize(s);
    if (e == cudaSuccess) swap(b);
    return e;
  }

  T *get() const { return p_; }
  operator T *() const { return p_; }
  T *operator->() const { return p_; }
  size_t size() const { return n_; }

 private:
  void swap(FbBuf &o) noexcept { std::swap(p_, o.p_); std::swap(n_, o.n_); }
  T *p_ = nullptr;
  size_t n_ = 0;
};

template <typename T> using FbDev = FbBuf<T, false>;
template <typename T> using FbPinned = FbBuf<T, true>;
