// Inline-PTX primitives shared by the forward and decode kernels.  Each one is defined here once, next to the stand-in the CPU
// emulator (tests/emu, built with HQQ_EMU) runs in its place.  The tcgen05 / mbarrier / TMA / TMEM wrappers are used by the
// tcgen05 GEMM alone and live in linear_gemm.cu.
#pragma once
#include <type_traits>

#include "common.cuh"

namespace hqq {

// ---- programmatic dependent launch (the emulator runs kernels one after another: nothing to wait for) ---------------
__device__ __forceinline__ void pdl_wait() {
#ifndef HQQ_EMU
  asm volatile("griddepcontrol.wait;" ::: "memory");
#endif
}
__device__ __forceinline__ void pdl_launch_dependents() {
#ifndef HQQ_EMU
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
#endif
}

// ---- bit manipulation ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t s) {
#ifdef HQQ_EMU
  return ::emu::prmt(a, b, s);
#else
  uint32_t r;
  asm("prmt.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(s));
  return r;
#endif
}
template <int LUT>
__device__ __forceinline__ uint32_t lop3(uint32_t a, uint32_t b, uint32_t c) {
#ifdef HQQ_EMU
  return ::emu::lop3(a, b, c, (uint32_t)LUT);
#else
  uint32_t r;
  asm("lop3.b32 %0, %1, %2, %3, %4;" : "=r"(r) : "r"(a), "r"(b), "r"(c), "n"(LUT));
  return r;
#endif
}

// ---- cp.async: 16-byte global -> shared copies in commit groups (the emulator lands a group at the wait that covers it) --
__device__ __forceinline__ void cp_async16(void* smem, const void* g) {
#ifdef HQQ_EMU
  ::emu::cp_async(smem, g, 16);
#else
  const uint32_t s = (uint32_t)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(s), "l"(g) : "memory");
#endif
}
__device__ __forceinline__ void cp_async_commit() {
#ifdef HQQ_EMU
  ::emu::cp_async_commit();
#else
  asm volatile("cp.async.commit_group;" ::: "memory");
#endif
}
template <int N>
__device__ __forceinline__ void cp_async_wait() {
#ifdef HQQ_EMU
  ::emu::cp_async_wait(N);
#else
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
#endif
}

// ---- system-scope relaxed accesses: the tagged words other kernels or peer GPUs write while this one polls them ------
__device__ __forceinline__ uint32_t ld_relaxed_sys_u32(const uint32_t* p) {
#ifdef HQQ_EMU
  return *reinterpret_cast<const volatile uint32_t*>(p);
#else
  uint32_t v;
  asm volatile("ld.relaxed.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
#endif
}
__device__ __forceinline__ uint4 ld_relaxed_sys_v4(const uint32_t* p) {
  uint4 v;
#ifdef HQQ_EMU
  memcpy(&v, p, 16);
#else
  asm volatile("ld.relaxed.sys.global.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p) : "memory");
#endif
  return v;
}
__device__ __forceinline__ void st_relaxed_sys_u32(uint32_t* p, uint32_t v) {
#ifdef HQQ_EMU
  *reinterpret_cast<volatile uint32_t*>(p) = v;
#else
  asm volatile("st.relaxed.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
#endif
}

__device__ __forceinline__ void prefetch_l2(const void* p) {
#ifndef HQQ_EMU
  asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
#endif
}

// ---- d = A[16x16] * B[16x8] + (zero_c ? 0 : d), fp32 accumulate: mma.sync with register fragments ---------------------
// zero_c takes C from a zero operand, so no instructions clear d first.
#define HQQ_MMA_M16N8K16(TY)                                                                                                      \
  if (zero_c)                                                                                                                     \
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32." TY "." TY ".f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%10,%10,%10,%10};" \
                 : "=f"(d[0]), "=f"(d[1]), "=f"(d[2]), "=f"(d[3])                                                                 \
                 : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1), "f"(0.0f));                                              \
  else                                                                                                                            \
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32." TY "." TY ".f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"     \
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])                                                                 \
                 : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1))
template <typename T>
__device__ __forceinline__ void mma_m16n8k16(float (&d)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1,
                                             bool zero_c) {
#ifdef HQQ_EMU
  ::emu::mma_m16n8k16<T>(d, a0, a1, a2, a3, b0, b1, zero_c);
#else
  static_assert(std::is_same<T, __half>::value || std::is_same<T, __nv_bfloat16>::value, "fp16 or bf16 operands");
  if constexpr (std::is_same<T, __half>::value) {
    HQQ_MMA_M16N8K16("f16");
  } else {
    HQQ_MMA_M16N8K16("bf16");
  }
#endif
}
#undef HQQ_MMA_M16N8K16

}  // namespace hqq
