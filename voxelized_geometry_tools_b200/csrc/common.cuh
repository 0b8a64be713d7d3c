// Shared host-side plumbing for the C-ABI translation units: thread-local error text,
// CUDA error mapping and a scoped device switch.
#pragma once

#include <cuda_runtime.h>

#include <algorithm>
#include <condition_variable>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <mutex>

#include "../../include/vgt_b200.h"

namespace vgt_b200
{
// Defined in capi_common.cu.
// Counts the kernels this library has launched (process-wide; vgt_b200_kernel_launch_count()).
void NoteKernelLaunch();
void SetLastError(const char* format, ...);
int FailInvalid(const char* format, ...);
int FailDevice(const char* what, cudaError_t error);

// Restores the caller's current device on scope exit. The reference helper calls
// cudaSetDevice on every entry (cuda_voxelization_helpers.cu:672, 769-774); we do the same but
// put the caller's device back so a host framework (torch) is not surprised.
class ScopedDevice
{
public:
  explicit ScopedDevice(int device) : status_(cudaSuccess), previous_(-1)
  {
    status_ = cudaGetDevice(&previous_);
    if (status_ == cudaSuccess && previous_ != device)
    {
      status_ = cudaSetDevice(device);
      switched_ = (status_ == cudaSuccess);
    }
  }
  ~ScopedDevice()
  {
    if (switched_)
    {
      cudaSetDevice(previous_);
    }
  }
  cudaError_t Status() const { return status_; }

private:
  cudaError_t status_;
  int previous_;
  bool switched_ = false;
};

// Owning device allocation for the host-pointer entry points.
template <typename T>
class DeviceBuffer
{
public:
  DeviceBuffer() = default;
  DeviceBuffer(const DeviceBuffer&) = delete;
  DeviceBuffer& operator=(const DeviceBuffer&) = delete;
  ~DeviceBuffer() { Release(); }
  cudaError_t Allocate(int64_t count)
  {
    Release();
    if (count <= 0)
    {
      return cudaSuccess;
    }
    return cudaMalloc(reinterpret_cast<void**>(&ptr_), sizeof(T) * static_cast<size_t>(count));
  }
  void Release()
  {
    if (ptr_ != nullptr)
    {
      cudaFree(ptr_);
      ptr_ = nullptr;
    }
  }
  T* get() const { return ptr_; }

private:
  T* ptr_ = nullptr;
};

// ------------------------------------------------------------------------------------------------
// Stream-ordered scratch. The default memory pool keeps freed blocks (release threshold raised
// once per device), so steady-state calls do not touch the OS allocator.
// ------------------------------------------------------------------------------------------------
inline void KeepPoolMemory(int device)
{
  static std::once_flag flags[64];
  if (device < 0 || device >= 64)
  {
    return;
  }
  std::call_once(flags[device], [device]()
  {
    cudaMemPool_t pool = nullptr;
    if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess)
    {
      unsigned long long threshold = ~0ull;
      cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &threshold);
    }
    cudaGetLastError();
  });
}

template <typename T>
class StreamScratch
{
public:
  StreamScratch() = default;
  StreamScratch(const StreamScratch&) = delete;
  StreamScratch& operator=(const StreamScratch&) = delete;
  ~StreamScratch()
  {
    if (ptr_ != nullptr)
    {
      cudaFreeAsync(ptr_, stream_);
    }
  }
  cudaError_t Allocate(int64_t count, cudaStream_t stream)
  {
    stream_ = stream;
    return cudaMallocAsync(reinterpret_cast<void**>(&ptr_), sizeof(T) * static_cast<size_t>(count),
                           stream);
  }
  T* get() const { return ptr_; }

private:
  T* ptr_ = nullptr;
  cudaStream_t stream_ = nullptr;
};

// Owns a stream created by the entry point (destroyed on scope exit).
struct StreamGuard
{
  cudaStream_t stream = nullptr;
  ~StreamGuard()
  {
    if (stream != nullptr)
    {
      cudaStreamDestroy(stream);
    }
  }
};

inline bool ValidDims(int64_t nx, int64_t ny, int64_t nz)
{
  return nx >= 1 && ny >= 1 && nz >= 1 && nx <= VGT_B200_MAX_AXIS && ny <= VGT_B200_MAX_AXIS
      && nz <= VGT_B200_MAX_AXIS;
}

// Part `index` of `total` items cut into `parts` near-equal parts (the first total % parts
// parts get one extra item): the x-slabs of the multi-device entries.
inline void SplitRange(int64_t total, int parts, int index, int64_t* begin, int64_t* end)
{
  const int64_t base = total / parts;
  const int64_t extra = total % parts;
  *begin = index * base + std::min<int64_t>(index, extra);
  *end = *begin + base + (index < extra ? 1 : 0);
}

// A reusable barrier for the per-device host threads (std::barrier is C++20).
class ThreadBarrier
{
public:
  explicit ThreadBarrier(int count) : count_(count), waiting_(0), generation_(0) {}
  void Wait()
  {
    std::unique_lock<std::mutex> lock(mutex_);
    const int generation = generation_;
    if (++waiting_ == count_)
    {
      waiting_ = 0;
      generation_++;
      released_.notify_all();
      return;
    }
    released_.wait(lock, [&] { return generation != generation_; });
  }

private:
  std::mutex mutex_;
  std::condition_variable released_;
  int count_;
  int waiting_;
  int generation_;
};
}  // namespace vgt_b200

#define VGT_CUDA_TRY(expr, what)                           \
  do                                                       \
  {                                                        \
    const cudaError_t vgt_status__ = (expr);               \
    if (vgt_status__ != cudaSuccess)                       \
    {                                                      \
      return ::vgt_b200::FailDevice((what), vgt_status__); \
    }                                                      \
  } while (0)
