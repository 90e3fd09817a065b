// txh_device.cuh -- inline-PTX device primitives of the routing and assimilation kernels (sm_100a), one name per
// instruction.  Shared-memory operands are 32-bit shared-window addresses (__cvta_generic_to_shared): no generic-address
// arithmetic in the loops.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>

#include "txh_kernels.cuh"

namespace txh {

// ---- global memory ----------------------------------------------------------------------------------------------
__device__ __forceinline__ int ld_relaxed_s32(const int* p)
{
    int v;
    asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ double ld_relaxed_f64(const double* p)
{
    double v;
    asm volatile("ld.relaxed.gpu.global.f64 %0, [%1];" : "=d"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ double2 ld_relaxed_row(const double* p)
{
    double2 v;
    asm volatile("ld.relaxed.gpu.global.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "l"(p) : "memory");
    return v;
}
// state rows are produced and consumed by different SMs inside one launch: bypass L1
__device__ __forceinline__ double2 ld_row(const double* p) { return __ldcg(reinterpret_cast<const double2*>(p)); }
__device__ __forceinline__ void st_row(double* p, double2 v) { __stcg(reinterpret_cast<double2*>(p), v); }

// ---- shared memory ----------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned lds_u16(unsigned sa)
{
    unsigned short v;
    asm volatile("ld.shared.u16 %0, [%1];" : "=h"(v) : "r"(sa));
    return v;
}
__device__ __forceinline__ uint32_t lds_u32(unsigned sa)
{
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(sa));
    return v;
}
__device__ __forceinline__ double lds_f64(unsigned sa)
{
    double v;
    asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(sa));
    return v;
}
__device__ __forceinline__ double2 lds_row(unsigned sa)
{
    double2 v;
    asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "r"(sa));
    return v;
}
__device__ __forceinline__ int4 lds_i4(unsigned sa)
{
    int4 v;
    asm volatile("ld.shared.v4.s32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(sa));
    return v;
}
__device__ __forceinline__ void sts_u16(unsigned sa, unsigned v)
{
    asm volatile("st.shared.u16 [%0], %1;" ::"r"(sa), "h"((unsigned short)v) : "memory");
}
__device__ __forceinline__ void sts_u32(unsigned sa, uint32_t v)
{
    asm volatile("st.shared.u32 [%0], %1;" ::"r"(sa), "r"(v) : "memory");
}
__device__ __forceinline__ void sts_f64(unsigned sa, double v)
{
    asm volatile("st.shared.f64 [%0], %1;" ::"r"(sa), "d"(v) : "memory");
}
__device__ __forceinline__ void sts_row(unsigned sa, double2 v)
{
    asm volatile("st.shared.v2.f64 [%0], {%1, %2};" ::"r"(sa), "d"(v.x), "d"(v.y) : "memory");
}
__device__ __forceinline__ void sts_i4(unsigned sa, int4 v)
{
    asm volatile("st.shared.v4.s32 [%0], {%1, %2, %3, %4};" ::"r"(sa), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

// ---- asynchronous global -> shared copies (LDGSTS); 16-byte copies bypass L1 ----------------------------------------
__device__ __forceinline__ void cp_async4(unsigned sa, const void* g)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(sa), "l"(g) : "memory");
}
__device__ __forceinline__ void cp_async8(unsigned sa, const void* g)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(sa), "l"(g) : "memory");
}
__device__ __forceinline__ void cp_async16(unsigned sa, const void* g)
{
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sa), "l"(g) : "memory");
}
// ... to a generic pointer into shared memory, converted once both operands are formed (converting at the call orders
// the address arithmetic differently)
__device__ __forceinline__ void cp_async4(void* s, const void* g) { cp_async4((unsigned)__cvta_generic_to_shared(s), g); }
__device__ __forceinline__ void cp_async8(void* s, const void* g) { cp_async8((unsigned)__cvta_generic_to_shared(s), g); }
__device__ __forceinline__ void cp_async16(void* s, const void* g) { cp_async16((unsigned)__cvta_generic_to_shared(s), g); }
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait_group() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// ---- special registers ------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long globaltimer_ns()
{
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
__device__ __forceinline__ unsigned smid()
{
    unsigned v;
    asm volatile("mov.u32 %0, %%smid;" : "=r"(v));
    return v;
}

// ---- programmatic dependent launch --------------------------------------------------------------------------------
// A kernel launched with cudaLaunchAttributeProgrammaticStreamSerialization may start once every CTA of the kernel
// before it in the stream has executed launch_dependents (or exited); what that kernel wrote is only visible after wait.
__device__ __forceinline__ void griddep_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void griddep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// ---- FP64 tensor cores --------------------------------------------------------------------------------------------
// D(8x8) += A(8x4) * B(4x8).  Fragment ownership (lane = 4*g + t): a = A[g][t], b = B[t][g], c0 = C[g][2t], c1 = C[g][2t+1]
__device__ __forceinline__ void dmma8x8x4(double& c0, double& c1, double a, double b)
{
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

// ---- EMPTY: the hand-over protocol of the rings of the persistent routing kernels (txh_window.cu, txh_lane.cu) -----
// A ring cell that has not been written holds every bit set (kEmptyByte in each byte, the fill of the host): a NaN no
// arithmetic produces.  The producer just stores its value; the consumer polls its own cell until it is not EMPTY and
// puts EMPTY back (every cell has exactly one reader), so a ring is clean again when a launch ends.
constexpr long long kEmptyBits = -1ll;
__device__ __forceinline__ bool is_empty(double v) { return __double_as_longlong(v) == kEmptyBits; }
__device__ __forceinline__ double empty_f64() { return __longlong_as_double(kEmptyBits); }
__device__ __forceinline__ double2 empty_row() { return make_double2(empty_f64(), empty_f64()); }
// both member columns of a 16-byte cell written
__device__ __forceinline__ bool cell_full(double2 v) { return !is_empty(v.x) && !is_empty(v.y); }

}  // namespace txh
