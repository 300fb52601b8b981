// evg_tcgen05.cuh — the 5th-generation tensor-core plumbing (tcgen05 MMAs into TMEM, mbarriers, bulk copies, the
// 128-byte-swizzled K-major operand layout) shared by the fused policy kernels evg_policy_mlp.cu and evg_policy_ppo.cu.
#pragma once
#include <cuda_bf16.h>
#include <stdint.h>

namespace evg {

constexpr int kAtomK = 64;  // bf16 elements in one 128-byte swizzle row

// K-major operand tile with 128-byte swizzle: element (row r, column k) of a [rows x K] bf16 matrix lives in atom k / 64
// (a block of rows x 128 bytes), at row r, 16-byte chunk ((k % 64) / 8) ^ (r % 8)
__host__ __device__ inline int swz_offset(int rows, int r, int k)
{
    return (k / kAtomK) * rows * 128 + r * 128 + ((((k % kAtomK) >> 3) ^ (r & 7)) << 4) + (k & 7) * 2;
}

#ifdef __CUDACC__
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): start address >> 4 [0:14), leading byte offset >> 4
// [16:30) (unused for a swizzled K-major operand), stride byte offset >> 4 [32:46) = 1024 B between 8-row groups,
// version 1 [46:48), layout SWIZZLE_128B = 2 [61:64)
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr)
{
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | (uint64_t)1 << 16 | (uint64_t)(1024 >> 4) << 32 | (uint64_t)1 << 46 | (uint64_t)2 << 61;
}

// instruction descriptor (cute::UMMA::InstrDescriptor): D fp32 [4:6) = 1, A bf16 [7:10) = 1, B bf16 [10:13) = 1, both
// K-major, N >> 3 at [17:23), M >> 4 at [24:29)
__device__ __forceinline__ uint32_t make_idesc(int m, int n)
{
    return 1u << 4 | 1u << 7 | 1u << 10 | (uint32_t)(n >> 3) << 17 | (uint32_t)(m >> 4) << 24;
}

__device__ __forceinline__ void umma(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate)
{
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accumulate)
        : "memory");
}

__device__ __forceinline__ void umma_commit(uint64_t* bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// wait for phase `parity` of an mbarrier; a bounded spin that traps instead of hanging the GPU if the MMAs never arrive
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity)
{
    const uint32_t a = smem_u32(bar);
    for (uint32_t spin = 0;; ++spin) {
        uint32_t done;
        asm volatile(
            "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}\n"
            : "=r"(done)
            : "r"(a), "r"(parity)
            : "memory");
        if (done) return;
        if (spin > (1u << 26)) __trap();
    }
}

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16])
{
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]),
          "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr));
}

__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi)
{
    const __nv_bfloat162 p = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<const uint32_t*>(&p);
}

// one bulk copy global -> shared memory, completion counted in bytes on `bar`
__device__ __forceinline__ void bulk_load(void* dst, const void* src, uint32_t bytes, uint64_t* bar)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)), "l"(src), "r"(bytes),
                 "r"(smem_u32(bar))
                 : "memory");
}
#endif

}  // namespace evg
