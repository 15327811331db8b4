// Shared helpers for the hqq_b200 sm_100a kernels.
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <atomic>

#include "../../include/hqq_b200.h"

namespace hqq {

// ---- error plumbing -----------------------------------------------------------------
void set_error(const char* fmt, ...);
extern std::atomic<long long> g_launches;
extern std::atomic<int> g_env_epoch;  // bumped by hqq_b200_reload_env(): cached HQQ_B200_* knobs are parsed again

// `static int var`, parsed from the environment by `expr` on first use and again after every hqq_b200_reload_env()
#define HQQ_ENV_KNOB(var, expr)                                                     \
  static int var = 0;                                                               \
  {                                                                                 \
    static int epoch__ = -1;                                                        \
    const int now__ = ::hqq::g_env_epoch.load(std::memory_order_relaxed);           \
    if (epoch__ != now__) { var = (expr); epoch__ = now__; }                        \
  }

#define HQQ_REQUIRE(cond, code, ...)            \
  do {                                          \
    if (!(cond)) {                              \
      ::hqq::set_error(__VA_ARGS__);            \
      return (code);                            \
    }                                           \
  } while (0)

// Launch check that is legal under stream capture (no sync).
#define HQQ_LAUNCH_CHECK(name)                                                 \
  do {                                                                         \
    cudaError_t e__ = cudaGetLastError();                                      \
    ::hqq::g_launches.fetch_add(1, std::memory_order_relaxed);                 \
    if (e__ != cudaSuccess) {                                                  \
      ::hqq::set_error("%s: CUDA launch failed: %s", name, cudaGetErrorString(e__)); \
      return HQQ_E_CUDA;                                                       \
    }                                                                          \
  } while (0)

static inline bool aligned(const void* p, size_t a) { return (reinterpret_cast<uintptr_t>(p) % a) == 0; }
static inline int64_t cdiv(int64_t a, int64_t b) { return (a + b - 1) / b; }

constexpr int kNumSMs = 148;  // B200

// ---- kernel launches ------------------------------------------------------------------
// Function attributes (opt-in dynamic shared memory) and SM counts belong to ONE device: the caches below are indexed by the
// calling thread's current device, so layers living on several GPUs of one process each get their own setup.
constexpr int kMaxDevices = 64;
int cur_device();   // the calling thread's current device (0 if it cannot be told)
int sm_count();     // SMs of the current device
bool pdl_enabled(); // false under HQQ_B200_PDL=0 (test hook): the linear kernels launch without programmatic dependent launch

// Raises kernel K's dynamic shared-memory limit on the current device to at least `bytes`.
template <auto K>
int reserve_smem(int bytes) {
  static int have[kMaxDevices] = {};
  int& h = have[cur_device()];
  if (bytes > h) {
    const cudaError_t e = cudaFuncSetAttribute(K, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    HQQ_REQUIRE(e == cudaSuccess, HQQ_E_CUDA, "hqq_b200_linear_fwd: cannot reserve %d bytes of shared memory: %s", bytes, cudaGetErrorString(e));
    h = bytes;
  }
  return HQQ_OK;
}

// Counted launch, with the programmatic-stream-serialization attribute when `pdl` is set: the kernel may become resident
// while its predecessor on the stream is still running, and waits for it in griddepcontrol.wait (pdl_wait).
template <typename K, typename... Args>
int launch_pdl(const char* name, K kernel, dim3 grid, dim3 block, size_t smem, cudaStream_t st, bool pdl, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = pdl ? 1 : 0;
  const cudaError_t e = cudaLaunchKernelEx(&cfg, kernel, args...);
  g_launches.fetch_add(1, std::memory_order_relaxed);
  HQQ_REQUIRE(e == cudaSuccess, HQQ_E_CUDA, "%s: CUDA launch failed: %s", name, cudaGetErrorString(e));
  return HQQ_OK;
}

static inline int fields_of(int nbits) { return nbits == 3 ? 10 : 8 / nbits; }
static inline bool valid_nbits(int nbits) { return nbits == 8 || nbits == 4 || nbits == 3 || nbits == 2 || nbits == 1; }
static inline size_t dtype_size(int dt) {
  switch (dt) {
    case HQQ_F32: case HQQ_I32: return 4;
    case HQQ_F16: case HQQ_BF16: return 2;
    case HQQ_U8: return 1;
    case HQQ_I64: return 8;
  }
  return 0;
}

// ---- device-side scalar conversions ---------------------------------------------------
template <typename T> __device__ __forceinline__ float to_f32(T v);
template <> __device__ __forceinline__ float to_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ float to_f32<__half>(__half v) { return __half2float(v); }
template <> __device__ __forceinline__ float to_f32<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }

template <typename T> __device__ __forceinline__ T from_f32(float v);
template <> __device__ __forceinline__ __half from_f32<__half>(float v) { return __float2half_rn(v); }
template <> __device__ __forceinline__ __nv_bfloat16 from_f32<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }

// integer level -> T (levels are < 256: exact in every type)
template <typename T> __device__ __forceinline__ T level_to(unsigned q);
template <> __device__ __forceinline__ float level_to<float>(unsigned q) { return (float)q; }
template <> __device__ __forceinline__ __half level_to<__half>(unsigned q) { return __ushort2half_rn((unsigned short)q); }
template <> __device__ __forceinline__ __nv_bfloat16 level_to<__nv_bfloat16>(unsigned q) { return __ushort2bfloat16_rn((unsigned short)q); }
template <> __device__ __forceinline__ uint8_t level_to<uint8_t>(unsigned q) { return (uint8_t)q; }
template <> __device__ __forceinline__ int32_t level_to<int32_t>(unsigned q) { return (int32_t)q; }
template <> __device__ __forceinline__ int64_t level_to<int64_t>(unsigned q) { return (int64_t)q; }

// (q - z) * s with one rounding per operation in T -- the reference's two-rounding dequant
// (hqq/core/quantize.py:198).  __fsub_rn/__fmul_rn forbid FMA contraction.
template <typename T> __device__ __forceinline__ T dequant_one(unsigned q, T z, T s);
template <> __device__ __forceinline__ float dequant_one<float>(unsigned q, float z, float s) {
  return __fmul_rn(__fsub_rn((float)q, z), s);
}
template <> __device__ __forceinline__ __half dequant_one<__half>(unsigned q, __half z, __half s) {
  return __hmul(__hsub(level_to<__half>(q), z), s);
}
template <> __device__ __forceinline__ __nv_bfloat16 dequant_one<__nv_bfloat16>(unsigned q, __nv_bfloat16 z, __nv_bfloat16 s) {
  return __hmul(__hsub(level_to<__nv_bfloat16>(q), z), s);
}

// ---- vector of N elements of T with 16/8/4-byte aligned storage ------------------------
template <typename T, int N>
struct alignas(sizeof(T) * N >= 16 ? 16 : sizeof(T) * N) Vec {
  T v[N];
};

// streaming 16-byte global load that does not pollute L1 (weights are read exactly once)
__device__ __forceinline__ uint4 ldg_stream_v4(const void* p) {
#ifdef HQQ_EMU
  return *reinterpret_cast<const uint4*>(p);
#endif
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}

}  // namespace hqq
