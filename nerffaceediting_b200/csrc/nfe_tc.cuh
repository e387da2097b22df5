// tcgen05 / TMEM / mbarrier primitives for sm_100a, written as raw PTX (no CUTLASS dependency).
//
// Operand layouts used by the decoder GEMMs (all K-major, SWIZZLE_NONE "interleave" layout):
//   an operand tile of R rows x K bf16 is a grid of 8x8-element core matrices (8 rows x 16 bytes,
//   128 contiguous bytes); core matrix (r/8, k/8) lives at  (r/8)*SBO + (k/8)*LBO  bytes from the
//   tile start.  One tcgen05.mma.kind::f16 consumes K = 16 (two core matrices along K).
// Accumulators live in TMEM: D[m][n] (fp32) is lane m, column col0 + n.
#pragma once
#include <cuda_bf16.h>
#include <stdint.h>

namespace nfe { namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- shared-memory matrix descriptor (SWIZZLE_NONE, K-major) ----------------------------------
__device__ __forceinline__ uint64_t make_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes)
{
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);           // start address, 16-byte units
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;     // leading (K-direction) core-matrix stride
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;     // stride (row-group) core-matrix stride
    d |= (uint64_t)1 << 46;                               // descriptor version: Blackwell
    return d;                                             // base_offset 0, lbo_mode 0, layout SWIZZLE_NONE
}

// ---- instruction descriptor: kind::f16, bf16 x bf16 -> fp32, both operands K-major ------------
__host__ __device__ constexpr uint32_t make_idesc_bf16(int M, int N)
{
    return (1u << 4)                     // D format: f32
         | (1u << 7)                     // A format: bf16
         | (1u << 10)                    // B format: bf16
         | ((uint32_t)(N >> 3) << 17)    // N / 8
         | ((uint32_t)(M >> 4) << 24);   // M / 16
}

// D[tmem] (+)= A[smem] * B[smem]^T ; issued by ONE thread on behalf of the CTA
__device__ __forceinline__ void mma_bf16_ss(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, bool accumulate)
{
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}\n"
        :: "r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"((uint32_t)accumulate) : "memory");
}

// D[tmem] (+)= A[tmem] * B[smem]^T : the A operand (M rows = TMEM lanes, K along the columns, two 16-bit elements per 32-bit
// column) comes straight from tensor memory, where an epilogue put it with tcgen05.st
__device__ __forceinline__ void mma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc, bool accumulate)
{
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t"
        "}\n"
        :: "r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"((uint32_t)accumulate) : "memory");
}

// One lane of the (converged) warp.  MMA-issuing code keeps its control flow warp-uniform and predicates only the tcgen05
// instructions on this: inside a divergent `if (lane == 0)` region the compiler has to wrap every tcgen05.mma in an ELECT /
// R2UR.BROADCAST waterfall loop to get descriptors into uniform registers (~24 dependent instructions, ~180 cycles per MMA measured).
__device__ __forceinline__ bool elect_one()
{
    uint32_t pred;
    asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.b32 %0, 1, 0, P;\n\t}" : "=r"(pred));
    return pred != 0;
}

// all previously issued MMAs of this thread arrive on the mbarrier when they complete
__device__ __forceinline__ void mma_commit(uint64_t* mbar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(smem_u32(mbar)) : "memory");
}

// ---- TMEM allocation (one full warp) ----------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols)
{
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(smem_u32(dst_smem)), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols)
{
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(taddr), "r"(ncols) : "memory");
}

__device__ __forceinline__ void fence_before_sync() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_after_sync() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// make generic-proxy shared-memory writes visible to the async proxy (the tensor core's operand reads)
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---- TMEM -> registers: 16 consecutive fp32 columns of this thread's lane ---------------------
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16])
{
    uint32_t r[16];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// ---- registers -> TMEM (tcgen05.st): wait until this thread's stores have landed
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// ---- mbarrier ----------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* mbar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(mbar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint64_t* mbar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(smem_u32(mbar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* mbar, uint32_t parity)
{
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t"   // suspend-time hint: sleep in hardware, do not spin on issue slots
        "@p bra WAIT_DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "WAIT_DONE:\n\t"
        "}\n"
        :: "r"(smem_u32(mbar)), "r"(parity), "r"(0x989680u) : "memory");
}

// ---- bf16 split: x ~= hi + lo with hi = bf16(x), lo = bf16(x - hi) ------------------------------
__device__ __forceinline__ void split_bf16(float x, __nv_bfloat16& hi, __nv_bfloat16& lo)
{
    hi = __float2bfloat16_rn(x);
    lo = __float2bfloat16_rn(x - __bfloat162float(hi));
}

__device__ __forceinline__ uint32_t pack_bf16(__nv_bfloat16 a, __nv_bfloat16 b)
{
    return (uint32_t)__bfloat16_as_ushort(a) | ((uint32_t)__bfloat16_as_ushort(b) << 16);
}

}}  // namespace nfe::tc
