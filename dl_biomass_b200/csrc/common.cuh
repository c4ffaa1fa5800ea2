// Shared device/host helpers for libb2pn (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/b2pn.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libb2pn is written for sm_100a (B200) only"
#endif

#define B2PN_LAUNCH_CHECK()                         \
    do {                                            \
        cudaError_t e__ = cudaPeekAtLastError();    \
        if (e__ != cudaSuccess) return (int)e__;    \
    } while (0)

#define B2PN_CUDA(call)                             \
    do {                                            \
        cudaError_t e__ = (call);                   \
        if (e__ != cudaSuccess) return (int)e__;    \
    } while (0)

namespace b2pn {

typedef unsigned long long u64;

// number of kernels this library has enqueued (bench.py reports it as gpu_launches)
extern long long g_launches;
// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-(kernel, device) property: raise it once, not on every launch
// (invisible under CUDA graphs, but ~1 us of host time per launch in the eager, ragged-batch training loop).
// `slot`: one static per call site (per kernel instantiation): the largest size set so far per device.
struct SmemAttrSlot {
    int bytes[64];
};
template <class K>
static inline cudaError_t ensure_dynamic_smem(K kern, int bytes, SmemAttrSlot &slot)
{
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev >= 0 && dev < 64 && slot.bytes[dev] >= bytes) return cudaSuccess;
    e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e == cudaSuccess && dev >= 0 && dev < 64) slot.bytes[dev] = bytes;   // a racing first call sets the same value twice
    return e;
}

static inline void note_launch(int n = 1) { __atomic_fetch_add(&g_launches, (long long)n, __ATOMIC_RELAXED); }

// ---- packed fp32x2 arithmetic (Blackwell FADD2/FMUL2), each half rounded separately ----------
// NOTE: ptxas contracts mul.f32x2 + add.f32x2 into FFMA2 even with .rn, which would break the
// bit-exact distance contract, so only sub and mul are packed; the adds stay scalar __fadd_rn.
// tests/test_build.py asserts there is no FFMA in the grouping kernels' SASS.
__device__ __forceinline__ u64 pack2(float lo, float hi)
{
    u64 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ float lo32(u64 a)
{
    float lo, hi;
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(a));
    (void)hi;
    return lo;
}
__device__ __forceinline__ float hi32(u64 a)
{
    float lo, hi;
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(a));
    (void)lo;
    return hi;
}
__device__ __forceinline__ u64 sub2(u64 a, u64 b)
{
    u64 r;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ u64 mul2(u64 a, u64 b)
{
    u64 r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}

// squared distance of two packed points to one reference, canonical rounding order
__device__ __forceinline__ void dist2_pair(u64 x, u64 y, u64 z, u64 px, u64 py, u64 pz, float &d0, float &d1)
{
    const u64 sx = sub2(x, px), sy = sub2(y, py), sz = sub2(z, pz);
    const u64 qx = mul2(sx, sx), qy = mul2(sy, sy), qz = mul2(sz, sz);
    d0 = __fadd_rn(__fadd_rn(lo32(qx), lo32(qy)), lo32(qz));
    d1 = __fadd_rn(__fadd_rn(hi32(qx), hi32(qy)), hi32(qz));
}

__device__ __forceinline__ float dist2_scalar(float x, float y, float z, float px, float py, float pz)
{
    const float dx = __fsub_rn(x, px), dy = __fsub_rn(y, py), dz = __fsub_rn(z, pz);
    return __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
}

// ---- cluster helpers ----------------------------------------------------------------------------
__device__ __forceinline__ unsigned cluster_ctarank()
{
    unsigned r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_arrive_release()
{
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
}
__device__ __forceinline__ void cluster_wait_acquire()
{
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ unsigned smem_u32(const void *p)
{
    return (unsigned)__cvta_generic_to_shared(p);
}
// map a local shared address to the same offset in CTA `rank` of the cluster
__device__ __forceinline__ unsigned mapa_u32(unsigned local_addr, unsigned rank)
{
    unsigned r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_addr), "r"(rank));
    return r;
}
__device__ __forceinline__ void st_cluster_v4(unsigned addr, unsigned a, unsigned b, unsigned c, unsigned d)
{
    asm volatile("st.shared::cluster.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d)
                 : "memory");
}
__device__ __forceinline__ void st_cluster_v2(unsigned addr, unsigned a, unsigned b)
{
    asm volatile("st.shared::cluster.v2.u32 [%0], {%1, %2};" ::"r"(addr), "r"(a), "r"(b) : "memory");
}

}  // namespace b2pn
