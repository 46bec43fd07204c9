// Shared host/device helpers for libhipac_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <string>
#include <utility>

#include "../../include/hipac_b200.h"

namespace hipac {

void set_error(const std::string& msg);
void count_launch(int n = 1);

// RAII CUDA-event bracket around one kernel launch; a no-op unless hipac_profile_enable(1).
class ProfileScope {
 public:
  ProfileScope(const char* name, cudaStream_t stream, double work = 0.0);
  ~ProfileScope();
 private:
  int idx_;
  cudaStream_t stream_;
};

#define HIPAC_CHECK_CUDA(expr)                                                              \
  do {                                                                                      \
    cudaError_t _e = (expr);                                                                \
    if (_e != cudaSuccess) {                                                                \
      ::hipac::set_error(std::string(#expr) + " failed: " + cudaGetErrorString(_e) + " (" + \
                         __FILE__ + ":" + std::to_string(__LINE__) + ")");                  \
      return -2;                                                                            \
    }                                                                                       \
  } while (0)

#define HIPAC_REQUIRE(cond, msg)                                     \
  do {                                                               \
    if (!(cond)) {                                                   \
      ::hipac::set_error(std::string("invalid argument: ") + (msg)); \
      return -1;                                                     \
    }                                                                \
  } while (0)

static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// Per-DEVICE one-time state (several GPUs may be driven from one process, from several threads):
//   ensure_dyn_smem  cudaFuncAttributeMaxDynamicSharedMemorySize is a per-device attribute of a kernel
//   device_sm_count  SM count of the current device
int ensure_dyn_smem_impl(const void* func, int bytes);
template <typename F>
static inline int ensure_dyn_smem(F* func, int bytes) { return ensure_dyn_smem_impl(reinterpret_cast<const void*>(func), bytes); }
int device_sm_count(int* sms);

// Launch with optional thread-block cluster and programmatic stream serialization (see ptx::pdl_wait in umma.cuh).
template <typename... KArgs, typename... Args>
static inline cudaError_t launch_ex(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, int cluster_x,
                                    Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid, cfg.blockDim = block, cfg.dynamicSmemBytes = smem, cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  int na = 0;
  if (cluster_x > 1) {
    attr[na].id = cudaLaunchAttributeClusterDimension;
    attr[na].val.clusterDim.x = (unsigned)cluster_x, attr[na].val.clusterDim.y = 1, attr[na].val.clusterDim.z = 1;
    na++;
  }
  attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[na].val.programmaticStreamSerializationAllowed = 1;
  na++;
  cfg.attrs = attr, cfg.numAttrs = (unsigned)na;
  return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}

// Device-side bounds assertions of the stage-1 kernels (compute-sanitizer is not available on the B200 pool): compiled
// in only with -DHIPAC_DEBUG_BOUNDS (libhipac_b200_dbg.so, exercised by tests/test_debug_bounds_gpu.py).
#ifdef HIPAC_DEBUG_BOUNDS
#define HIPAC_DEV_ASSERT(cond)                                                                             \
  do {                                                                                                     \
    if (!(cond)) {                                                                                         \
      printf("hipac bounds assertion failed: %s (%s:%d, block %d thread %d)\n", #cond, __FILE__, __LINE__, \
             (int)blockIdx.x, (int)threadIdx.x);                                                           \
      __trap();                                                                                            \
    }                                                                                                      \
  } while (0)
#else
#define HIPAC_DEV_ASSERT(cond) ((void)0)
#endif

constexpr int OUT = 224;  // network input size (reference src/main.py:814)

}  // namespace hipac
