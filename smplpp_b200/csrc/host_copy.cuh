// Host-side helpers of the host-buffer pipelines (host_pipe.cu: smplpp_forward_host, task_forward.cu:
// smplpp_task_forward_host): page-lock detection, multi-threaded host copies into / out of pinned staging buffers and
// grow-only device / pinned allocations.
#pragma once
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <thread>

#include "common.cuh"

namespace sb
{
inline bool is_page_locked(const void * p)
{
  cudaPointerAttributes attr;
  if(cudaPointerGetAttributes(&attr, p) != cudaSuccess)
  {
    cudaGetLastError();
    return false;
  }
  return attr.type == cudaMemoryTypeHost;
}

// dst <- src on up to `threads` host threads (a single thread moves ~10 GB/s, the link ~55 GB/s)
inline void parallel_memcpy(void * dst, const void * src, size_t bytes, int threads)
{
  constexpr size_t kMinPerThread = 1 << 20;
  threads = static_cast<int>(std::max<size_t>(1, std::min<size_t>(threads, bytes / kMinPerThread)));
  if(threads == 1)
  {
    memcpy(dst, src, bytes);
    return;
  }
  const size_t per = align_up((bytes + threads - 1) / threads, 4096);
  std::thread pool[16];
  int started = 0;
  for(int t = 0; t < threads; t++)
  {
    const size_t off = per * t;
    if(off >= bytes) break;
    const size_t n = std::min(per, bytes - off);
    pool[started++] = std::thread([=] { memcpy(static_cast<char *>(dst) + off, static_cast<const char *>(src) + off, n); });
  }
  for(int t = 0; t < started; t++) pool[t].join();
}

inline int host_threads()
{
  static int n = 0;
  if(n == 0)
  {
    const char * e = getenv("SMPLPP_HOST_THREADS");
    n = e ? atoi(e) : static_cast<int>(std::thread::hardware_concurrency() / 2);
    n = std::max(1, std::min(n, 16));
  }
  return n;
}

inline int grow_dev(void ** p, size_t * have, size_t need)
{
  if(*have >= need) return SMPLPP_OK;
  if(*p) cudaFree(*p);
  *p = nullptr;
  *have = 0;
  SB_CUDA(cudaMalloc(p, need));
  *have = need;
  return SMPLPP_OK;
}

inline int grow_pinned(void ** p, size_t * have, size_t need)
{
  if(*have >= need) return SMPLPP_OK;
  if(*p) cudaFreeHost(*p);
  *p = nullptr;
  *have = 0;
  SB_CUDA(cudaHostAlloc(p, need, cudaHostAllocPortable));
  *have = need;
  return SMPLPP_OK;
}
} // namespace sb
