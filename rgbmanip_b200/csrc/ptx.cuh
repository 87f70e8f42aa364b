// PTX wrappers shared by the tcgen05 kernels (sm_100a): mbarrier, TMA, TMEM, tcgen05.mma / ld / commit.
#pragma once
#include "common.cuh"

namespace adp {

// ------------------------------------------------------------------------------------------------
// PTX wrappers (sm_100a)
// ------------------------------------------------------------------------------------------------
namespace ptx {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok != 0;
}
// Bounded wait: a pipeline bug must end in a trapped kernel with a flag, never in a hung GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity, int* err, int code) {
    if (mbar_try_wait(bar, parity)) return;
    long long t0 = clock64();
    while (!mbar_try_wait(bar, parity)) {
        if (clock64() - t0 > 4000000000LL) {
            if (err) atomicExch(err, code);
            __threadfence_system();
            asm volatile("trap;");
        }
    }
}

__device__ __forceinline__ void tma_load_5d(const CUtensorMap* map, uint32_t bar, uint32_t dst, int c0, int c1, int c2,
                                            int c3, int c4) {
    asm volatile(
        "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes"
        " [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
        ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
        : "memory");
}
__device__ __forceinline__ void tma_load_4d(const CUtensorMap* map, uint32_t bar, uint32_t dst, int c0, int c1, int c2, int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes"
        " [%0], [%1, {%3, %4, %5, %6}], [%2];"
        ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}
__device__ __forceinline__ void tma_load_3d(const CUtensorMap* map, uint32_t bar, uint32_t dst, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes"
        " [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}
// TMA store of a shared-memory box (bulk async group of the issuing thread): out-of-range elements of the box are not written
__device__ __forceinline__ void tma_store_5d(const CUtensorMap* map, uint32_t src, int c0, int c1, int c2, int c3, int c4) {
    asm volatile(
        "cp.async.bulk.tensor.5d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5, %6}], [%1];"
        ::"l"(reinterpret_cast<uint64_t>(map)), "r"(src), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
        : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }   // sources reusable
__device__ __forceinline__ void bulk_wait0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }             // writes complete
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}

__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem] * B[smem], bf16 x bf16 -> fp32, issued by one thread for the CTA.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc)
        : "memory");
}
// Warp-convergent issue: every lane executes the surrounding code with identical (warp-uniform) operands and only the
// elected lane's instruction takes effect.  Inside an `if (lane == 0)` branch ptxas must assume divergent, per-lane operands
// and wraps every tcgen05.mma in an ELECT / R2UR.BROADCAST / BRA.U.ANY waterfall (~10 issue slots + a branch per MMA), which
// bounds small-N MMAs (16-32 cycles of tensor work each) by the issuing thread instead of the tensor pipe.
__device__ __forceinline__ uint32_t elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred;
}
__device__ __forceinline__ void umma_bf16_elected(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc,
                                                  uint32_t elected) {
    asm volatile(
        "{\n\t.reg .pred p, e;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "setp.ne.b32 e, %5, 0;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc), "r"(elected)
        : "memory");
}
// fp8 (e4m3 x e4m3 -> fp32) MMA, K = 32 per instruction: twice the rate of kind::f16
__device__ __forceinline__ void umma_f8_elected(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc,
                                                uint32_t elected) {
    asm volatile(
        "{\n\t.reg .pred p, e;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "setp.ne.b32 e, %5, 0;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::f8f6f4 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc), "r"(elected)
        : "memory");
}
// kind::f16 MMA with scale-input-d = 15: D = A B + D * 2^-15.  Joins an accumulator that was built with operands pre-scaled by
// 2^15 in total (the fp8 low-order pass) to the unscaled fp16 pass.
__device__ __forceinline__ void umma_f16_scale15_elected(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t elected) {
    asm volatile(
        "{\n\t.reg .pred p, e;\n\t"
        "setp.ne.b32 p, 1, 0;\n\t"
        "setp.ne.b32 e, %4, 0;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p, 15;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(elected)
        : "memory");
}
__device__ __forceinline__ void umma_commit_elected(uint32_t bar, uint32_t elected) {
    asm volatile(
        "{\n\t.reg .pred e;\n\tsetp.ne.b32 e, %1, 0;\n\t"
        "@e tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}" ::"r"(bar), "r"(elected) : "memory");
}
// mbarrier arrives once all tcgen05 ops previously issued by this thread have completed.
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t* r) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t* r) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

}  // namespace ptx

// Shared-memory matrix descriptor, K-major operand whose rows are KC*2 bytes (= the swizzle span).
//   [0,14) start >> 4 | [16,30) LBO >> 4 (unused for swizzled K-major) | [32,46) SBO >> 4 (8-row group pitch)
//   [46,48) version = 1 (sm_100) | [49,52) base offset = 0 (tiles are 1024B aligned) | [61,64) layout type
template <int KC>
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr) {
    constexpr uint64_t layout = (KC == 64) ? 2ull : (KC == 32) ? 4ull : 6ull;   // SWIZZLE_128B / 64B / 32B
    constexpr uint64_t sbo = (uint64_t)(8 * KC * 2) >> 4;
    return (uint64_t)((smem_addr & 0x3FFFF) >> 4) | (1ull << 16) | (sbo << 32) | (1ull << 46) | (layout << 61);
}
// K-major operand without swizzle: 8-row x 16-byte core matrices; LBO = byte distance between the two 16-byte K chunks of one
// MMA, SBO = byte distance between consecutive 8-row groups.
__device__ __forceinline__ uint64_t make_desc_noswz(uint32_t addr, uint32_t lbo, uint32_t sbo) {
    return (uint64_t)((addr & 0x3FFFF) >> 4) | ((uint64_t)(lbo >> 4) << 16) | ((uint64_t)(sbo >> 4) << 32) | (1ull << 46);
}

// Instruction descriptor for kind::f16: D = fp32, A = B = bf16 (or fp16), both K-major, M = 128, N = n.
__device__ __forceinline__ uint32_t make_idesc_n(int n, int f16) {
    const uint32_t fmt = f16 ? 0u : 1u;   // F16 = 0, BF16 = 1
    return (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
}

}  // namespace adp
