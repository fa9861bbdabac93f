// PTX wrappers shared by the three tcgen05 kernels (fused_tc.cu, gemm_path.cu, gram_tc.cu): mbarriers, TMA, tensor memory, the
// UMMA instruction and shared-memory descriptors, and the host lookup of cuTensorMapEncodeTiled.  Each bit layout lives here once.
// What stays with a kernel: its mbarrier wait loop (suspend hint, watchdog and debug trace differ per kernel; each calls
// mbar_try_wait) and the wrappers only that kernel uses.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace desmo {
namespace ptx {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ------------------------------------------------------------------------------------------------- mbarriers and TMA
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
// makes the mbarrier.init of this thread visible to the async proxy (TMA, tcgen05.commit) and to the other threads
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
// One try_wait on phase `parity`: 1 once it has completed.  While it is open the thread may be suspended for up to ~hint_ns first.
__device__ __forceinline__ uint32_t mbar_try_wait(uint32_t bar, uint32_t parity, uint32_t hint_ns) {
    uint32_t done;
    asm volatile("{\n\t.reg .pred q;\n\tmbarrier.try_wait.parity.shared::cta.b64 q, [%1], %2, %3;\n\tselp.u32 %0, 1, 0, q;\n\t}\n"
                 : "=r"(done) : "r"(bar), "r"(parity), "r"(hint_ns) : "memory");
    return done;
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                 ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(bar) : "memory");
}
// generic-proxy shared-memory stores -> visible to the async proxy (an MMA or TMA that reads them after the next hand-over)
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ bool elect_one_sync() {
    uint32_t pred = 0;
    asm volatile("{\n\t.reg .b32 rx;\n\t.reg .pred px;\n\telect.sync rx|px, %1;\n\t@px mov.s32 %0, 1;\n\t}\n" : "+r"(pred) : "r"(0xffffffffu));
    return pred != 0;
}

// ------------------------------------------------------------------------------------------------- tensor memory and MMA
// kCols TMEM columns (a power of two >= 32) for this CTA, base address written to shared memory at dst, and the CTA's permit to
// allocate again given up; one whole warp calls it, the same warp later calls tmem_dealloc
template <uint32_t kCols>
__device__ __forceinline__ void tmem_alloc(uint32_t dst) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst), "r"(kCols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <uint32_t kCols>
__device__ __forceinline__ void tmem_dealloc(uint32_t tmem) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(kCols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mma_bf16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
        ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t* v) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
                   "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
                 : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// instruction descriptor, kind::f16 with bf16 operands and fp32 accumulation; a_mn / b_mn = 1: that operand is MN-major
__host__ __device__ constexpr uint32_t make_idesc_bf16(int M, int N, int a_mn, int b_mn) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)a_mn << 15) | ((uint32_t)b_mn << 16) | ((uint32_t)(N >> 3) << 17) |
           ((uint32_t)(M >> 4) << 24);
}
// Shared-memory descriptor: the high word is constant per operand role; the low word is (addr >> 4) | (LBO >> 4) << 16, so stepping
// through planes / k-steps is one 32-bit add per operand (shared-memory addresses < 256 KB never carry out of 14 bits).
constexpr uint32_t kDescHi = (1024u >> 4) | (1u << 14) | (2u << 29);  // SBO = 1024 B, version 1, SWIZZLE_128B
__device__ __forceinline__ uint64_t desc_from(uint32_t lo, uint32_t hi) { return ((uint64_t)hi << 32) | lo; }

// ------------------------------------------------------------------------------------------------- host
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                  CUtensorMapFloatOOBfill);
// the driver's cuTensorMapEncodeTiled through the runtime (no link against libcuda); nullptr if the driver lacks it
inline EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess && qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}

}  // namespace ptx
}  // namespace desmo
