// tc_mlp.cuh — tcgen05 (5th-gen tensor core) building blocks for the policy's 18->256 layers (sm_100a only).
//
// One CTA drives one or two M = 128 tiles: A = observations [128 x K] and B = first-layer weights [256 x K]
// (K = 24: 18 inputs, a constant 1 that carries the bias, zero padding) are staged in shared memory in the
// canonical K-major, no-swizzle UMMA layout; D = A * B^T [128 x 256] float32 accumulates in tensor memory
// (one row per TMEM lane = one environment per thread on read-back).
//
// Shared-memory operand layout (CUTLASS mma_traits_sm100.hpp, Major-K / INTERLEAVE): 8-row x 16-byte core
// matrices, each stored as 128 contiguous bytes; K-adjacent core matrices LBO bytes apart, 8-row groups SBO
// bytes apart.  Here: element (row, k) lives at  (row/8)*SBO + (k/4)*LBO + (row%8)*16 + (k%4)*4.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace carenv {
namespace tc {

constexpr int kK = 24;                 // padded reduction size (3 MMAs of K = 8 for kind::tf32)
constexpr int kKChunks = kK / 4;       // 16-byte chunks per row
constexpr int kLBO = 128;              // bytes between K-adjacent core matrices
constexpr int kSBO = kKChunks * 128;   // bytes between 8-row groups (768)
constexpr int kTileM = 128, kTileN = 256;
constexpr int kABytes = kTileM * kK * 4;   // 12,288
constexpr int kBBytes = kTileN * kK * 4;   // 24,576

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ int operand_offset(int row, int k) {
    return (row >> 3) * kSBO + (k >> 2) * kLBO + (row & 7) * 16 + (k & 3) * 4;
}

// 64-bit shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): start address, LBO, SBO in 16-byte
// units, version 1 (Blackwell), no swizzle.
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);            // bits [0,14)
    d |= (uint64_t)(kLBO >> 4) << 16;                        // bits [16,30)
    d |= (uint64_t)(kSBO >> 4) << 32;                        // bits [32,46)
    d |= (uint64_t)1 << 46;                                  // version_ = 1
    return d;                                                // layout_type (bits [61,64)) = 0: SWIZZLE_NONE
}

// 32-bit instruction descriptor (cute::UMMA::InstrDescriptor): D = F32, A = B = TF32, both K-major, N, M.
__device__ __forceinline__ uint32_t make_idesc_tf32(int M, int N) {
    return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

__device__ __forceinline__ void mma_tf32(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                         bool accumulate) {
    const uint32_t acc = accumulate ? 1u : 0u;
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}\n"
        :: "r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(acc) : "memory");
}

__device__ __forceinline__ void mma_commit(uint32_t mbar_smem) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n"
                 :: "r"(mbar_smem) : "memory");
}

__device__ __forceinline__ void mbar_init(uint32_t mbar_smem, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" :: "r"(mbar_smem), "r"(count) : "memory");
}

__device__ __forceinline__ void mbar_arrive(uint32_t mbar_smem) {
    asm volatile("{\n\t.reg .b64 t;\n\tmbarrier.arrive.shared::cta.b64 t, [%0];\n\t}\n" :: "r"(mbar_smem) : "memory");
}

// Bounded wait: a wrong descriptor must not hang the GPU box — trap instead.
__device__ __forceinline__ void mbar_wait(uint32_t mbar_smem, uint32_t parity) {
    uint32_t done = 0;
    for (int spin = 0; spin < (1 << 26); ++spin) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}\n"
            : "=r"(done) : "r"(mbar_smem), "r"(parity) : "memory");
        if (done) return;
    }
    __trap();
}

__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory"); }

// One full warp allocates `cols` TMEM columns (power of two >= 32) and publishes the base address in smem.
template <int COLS>
__device__ __forceinline__ void tmem_alloc(uint32_t *slot_smem) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n"
                 :: "r"(smem_u32(slot_smem)), "n"(COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
}
template <int COLS>
__device__ __forceinline__ void tmem_dealloc(uint32_t base) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" :: "r"(base), "n"(COLS) : "memory");
}

// 16 consecutive float32 columns of this thread's TMEM lane (warp w reads lanes 32*(w%4) .. +31).
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
    uint32_t r[16];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr) : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

// Ordered 16-byte shared-memory load: volatile, so a hand-written software pipeline of loads keeps its order.
__device__ __forceinline__ float4 lds128(uint32_t smem_addr) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];\n" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(smem_addr));
    return v;
}

__device__ __forceinline__ float to_tf32(float x) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;\n" : "=r"(r) : "f"(x));
    return __uint_as_float(r);
}

}  // namespace tc
}  // namespace carenv
