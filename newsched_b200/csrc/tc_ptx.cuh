// tc_ptx.cuh -- tcgen05 / TMEM PTX wrappers shared by the tensor-core kernels (fir_tc.cu, pfb.cu).
#pragma once
#include <cuda_bf16.h>

#include "common.cuh"

namespace b200 {

// 1024-byte aligned start inside a dynamic shared-memory array.  The offset is computed from the 32-bit shared
// address and ADDED to the array, so the compiler keeps the shared address space of everything derived from it
// (LDS / STS with 32-bit addresses); rounding the generic pointer as an integer loses that and turns every
// access into a generic LD / ST with 64-bit address arithmetic.
__device__ __forceinline__ uint8_t* tc_align1024(uint8_t* raw)
{
    return raw + ((1024u - (smem_u32(raw) & 1023u)) & 1023u);
}

// ---- tcgen05 / TMEM PTX ------------------------------------------------------------------------
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_alloc(uint32_t* smem_dst, uint32_t ncols)
{
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tc_dealloc(uint32_t taddr, uint32_t ncols)
{
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// arrives on the mbarrier once every tcgen05.mma issued so far by this thread has completed
__device__ __forceinline__ void tc_commit(uint64_t* bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc]^T, bf16 operands, fp32 accumulate; issued by ONE thread
__device__ __forceinline__ void tc_mma_bf16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                            uint32_t accumulate)
{
    asm volatile("{\n"
                 ".reg .pred p;\n"
                 "setp.ne.b32 p, %4, 0;\n"
                 "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
                 "}\n" ::"r"(d_tmem),
                 "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
                 : "memory");
}
// one lane of a converged warp (CUTLASS's elect_one_sync): the predicate comes from elect.sync, which the
// compiler knows to be true for exactly one lane, so operands need no per-lane loop to reach the uniform registers
__device__ __forceinline__ uint32_t tc_elect_one()
{
    uint32_t pred = 0, laneid = 0;
    asm volatile("{\n"
                 ".reg .b32 %%rx;\n"
                 ".reg .pred %%px;\n"
                 "elect.sync %%rx|%%px, %2;\n"
                 "@%%px mov.s32 %1, 1;\n"
                 "mov.s32 %0, %%rx;\n"
                 "}\n"
                 : "+r"(laneid), "+r"(pred)
                 : "r"(0xFFFFFFFFu));
    return pred;
}
// warp index as a warp-uniform value for the compiler (a shuffle result is uniform by construction): keeps the
// role dispatch and everything computed under it in the uniform datapath
__device__ __forceinline__ int tc_warp_idx() { return __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0); }

// Whole-warp forms: every lane executes them with warp-uniform operands and ONE lane is elected inside
// the asm.  Issuing under `if (lane == 0)` makes the operands thread-divergent for the compiler, which
// then wraps every UTCHMMA in an ELECT / R2UR.BROADCAST / BRA.U.ANY loop (~75 ns per MMA measured);
// with uniform operands the descriptors live in uniform registers and an MMA is a handful of instructions.
__device__ __forceinline__ void tc_commit_w(uint32_t bar_saddr)
{
    asm volatile("{\n"
                 ".reg .pred e;\n"
                 "elect.sync _|e, 0xffffffff;\n"
                 "@e tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n"
                 "}\n" ::"r"(bar_saddr)
                 : "memory");
}
__device__ __forceinline__ void tc_mma_bf16_w(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                              uint32_t accumulate)
{
    asm volatile("{\n"
                 ".reg .pred p, e;\n"
                 "setp.ne.b32 p, %4, 0;\n"
                 "elect.sync _|e, 0xffffffff;\n"
                 "@e tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
                 "}\n" ::"r"(d_tmem),
                 "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
                 : "memory");
}
__device__ __forceinline__ void tc_mma_bf16_ts_w(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc,
                                                 uint32_t accumulate)
{
    asm volatile("{\n"
                 ".reg .pred p, e;\n"
                 "setp.ne.b32 p, %4, 0;\n"
                 "elect.sync _|e, 0xffffffff;\n"
                 "@e tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n"
                 "}\n" ::"r"(d_tmem),
                 "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(accumulate)
                 : "memory");
}
// 32 consecutive fp32 columns of this thread's TMEM lane
__device__ __forceinline__ void tc_ld32(uint32_t taddr, float (&v)[32])
{
    uint32_t* u = reinterpret_cast<uint32_t*>(v);
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                 "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                 "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                 : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7]),
                   "=r"(u[8]), "=r"(u[9]), "=r"(u[10]), "=r"(u[11]), "=r"(u[12]), "=r"(u[13]), "=r"(u[14]), "=r"(u[15]),
                   "=r"(u[16]), "=r"(u[17]), "=r"(u[18]), "=r"(u[19]), "=r"(u[20]), "=r"(u[21]), "=r"(u[22]), "=r"(u[23]),
                   "=r"(u[24]), "=r"(u[25]), "=r"(u[26]), "=r"(u[27]), "=r"(u[28]), "=r"(u[29]), "=r"(u[30]), "=r"(u[31])
                 : "r"(taddr)
                 : "memory");
}
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// shared-memory matrix descriptor, K-major, SWIZZLE_128B: rows at 128 bytes, 8-row groups at SBO = 1024
__device__ __forceinline__ uint64_t tc_desc(uint32_t saddr)
{
    uint64_t d = (uint64_t)((saddr >> 4) & 0x3FFF);
    d |= (uint64_t)1 << 16;            // leading byte offset (unused: a K-step lies inside one swizzle row)
    d |= (uint64_t)(1024 >> 4) << 32;  // stride byte offset between 8-row groups
    d |= (uint64_t)1 << 46;            // descriptor version (sm_100)
    d |= (uint64_t)2 << 61;            // SWIZZLE_128B
    return d;
}

// byte offset of element i of a plane (rows of 64 bf16, 16-byte chunks XOR-swizzled by row & 7)
__device__ __forceinline__ uint32_t tc_plane_off(uint32_t i)
{
    return (i >> 6) * 128u + ((((i >> 3) & 7u) ^ ((i >> 6) & 7u)) << 4) + (i & 7u) * 2u;
}

__device__ __forceinline__ void tc_split(float v, __nv_bfloat16& hi, __nv_bfloat16& lo)
{
    hi = __float2bfloat16_rn(v);
    lo = __float2bfloat16_rn(v - __bfloat162float(hi));
}

__device__ __forceinline__ void tc_mma_bf16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc,
                                               uint32_t accumulate)
{
    asm volatile("{\n"
                 ".reg .pred p;\n"
                 "setp.ne.b32 p, %4, 0;\n"
                 "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n"
                 "}\n" ::"r"(d_tmem),
                 "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(accumulate)
                 : "memory");
}
__device__ __forceinline__ void tc_st8(uint32_t taddr, const uint32_t (&v)[8])
{
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(v[0]),
                 "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
                 : "memory");
}

} // namespace b200
