// Fused residual + gradient pass on the 5th-gen tensor cores (DESMO_PATH_TC): tcgen05.mma kind::f16 with every fp32 operand
// split into bf16 terms (x = x1 + x2 + x3 carries all 24 significand bits; Rec = G W keeps the six products with i + j <= 4, so it
// is accurate to ~2^-24 relative, i.e. fp32-class, at the cost of 6 bf16 MMAs = 3 TF32-equivalents).
//
// One persistent CTA per SM; a CTA owns tiles of 128 mesh points and walks all snapshots in slabs of 128:
//   G1  Rec[p x t]    = G[p x lib] W[lib x t]           -> TMEM cols [0,128)   (A = the three G planes resident in TMEM)  (CYL:548,565-572)
//   epi r = Rec - U   (U read once from HBM through per-quarter TMA stages; R never leaves the SM) (CYL:722); sum r^2;
//       r -> two bf16 planes (formed in registers before R_s is free), then R_s[p rows][t contiguous] in shared memory
//       (128B-swizzled: K-major operand of G3 AND MN-major operand of G4)
//   G3  D[p x lib]   += R[p x t] W^T[t x lib]           -> TMEM cols [128,192): two N-stacked blocks, accumulated over the slabs
//   G4  E^T[t x lib] += R^T[t x p] G[p x lib]           -> TMEM cols [256+32*slab, +32), accumulated over the tiles of the CTA and
//       drained every 32 tiles into the CTA's fp32 partial (the tensor core truncates when it adds into the accumulator)
// Warp roles (20 warps): warp 0 = TMA producer (W slab planes, phi / P tiles), warp 1 = MMA issuer (one elected thread), warps 2-3 =
// TMA producers of U (warp 2 also allocates TMEM), warps 4..19 = epilogue: thread <-> (mesh point == TMEM lane, snapshot quarter h);
// warp e = 4 + 4h + q handles lane quadrant q and snapshots 32h..32h+31 of the slab.
// The MMA issuer always runs G1 of the next slab-tile ahead of G3/G4 of the current one -- across tile boundaries too: the library
// row of the NEXT tile is evaluated one term per slab in the epilogue's slack (phi / P arrive by TMA a tile ahead), its TMEM planes
// (A of G1) are written as soon as G1 of the current tile's last slab has completed, and its shared-memory planes (B of G4) are
// written lane quadrant by lane quadrant together with the first R_s of the new tile, when G4 has released that quadrant.
#include <cuda.h>
#include <stdlib.h>
#include <string.h>
#include <cuda_bf16.h>

#include <type_traits>

#include "common.cuh"

namespace desmo {

namespace tc {
constexpr int KP = 32;          // padded library size handled by this kernel
constexpr int BP = 128;         // points per tile  (MMA M of G1/G3, K of G4)
constexpr int BT = 128;         // snapshots per slab (MMA N of G1, K of G3, M of G4)
constexpr int MAXSLAB = 8;      // TMEM: 8 x 32 columns of E accumulators
constexpr int E_FLUSH_TILES = 32;  // the tensor core adds into fp32 accumulators with truncation: bound the chain length (bias ~1e-8 per MMA)
constexpr int EPI_WARPS = 16;      // 4 lane quadrants x 4 snapshot quarters
constexpr int EPI_THREADS = EPI_WARPS * 32;
constexpr int THREADS = 128 + EPI_THREADS;
#ifndef DESMO_SETMAXNREG
#define DESMO_SETMAXNREG 0
#endif
#ifndef DESMO_REGS_EPI
#define DESMO_REGS_EPI 112
#define DESMO_REGS_CTRL 32
#endif
constexpr int REGS_EPI = DESMO_REGS_EPI, REGS_CTRL = DESMO_REGS_CTRL;  // setmaxnreg budgets (per thread) of the epilogue / control warpgroups
constexpr int NQ = 4;              // snapshot quarters per slab
constexpr int QT = BT / NQ;        // 32 snapshots per epilogue thread
constexpr int TPT = KP / NQ;       // library terms evaluated per epilogue thread (the four quarters of a point share the row)
constexpr uint32_t R_PLANE = 2 * BP * 128;            // one bf16 plane of R: 2 boxes [128 p rows x 128 B (64 t)]
constexpr uint32_t W_BOX = 3 * KP * 128;              // W slab box: [3 planes x 32 lib rows][128 B = 64 t]; planes stacked along rows
constexpr uint32_t W_PLANE = KP * 128;                // row offset of a plane inside a box
constexpr uint32_t W_SLAB = 2 * W_BOX;                // two boxes (snapshots 0-63, 64-127)
constexpr uint32_t G_PLANE = 2 * KP * 128;            // one bf16 plane of G: 2 boxes [32 lib rows x 128 B (64 p)]
// Planes of R (and of the W / G operands that multiply it) used by the two gradient GEMMs G3 / G4.  Two bf16 planes carry 16
// significand bits; with the three products R1*X1 + R1*X2 + R2*X1 the gradients come out at ~3e-7 relative (measured against an
// fp64 evaluation on the golden cases: 2e-7 .. 1.4e-6, the same class as a plain fp32 GEMM), far inside the 1e-5 gate, while Rec = G W
// keeps all three planes (R is a small difference of large numbers).
constexpr int NPR = 2;
#ifndef DESMO_G4_COLLECT
#define DESMO_G4_COLLECT 1
#endif
#ifndef DESMO_G1_WS
#define DESMO_G1_WS 0
#endif
constexpr uint32_t R_OFF = 0;
constexpr uint32_t W_OFF = R_OFF + NPR * R_PLANE;
constexpr uint32_t G_OFF = W_OFF + 2 * W_SLAB;        // two planes (B of G4); G1 reads its three planes from TMEM
constexpr uint32_t LAT_OFF = G_OFF + 2 * G_PLANE;     // phi tile [kMaxR][128] then P tile [kMaxR][128] of the tile whose library is next
constexpr uint32_t LAT_HALF = kMaxR * BP * 4;
// U staging: each snapshot quarter of the epilogue owns a private ring of U_RING TMA stages of [U_ROWS snapshots][128 points] fp32
// (bf16 snapshots: the same stages at half the bytes, in the first half of the fp32-sized region).
// Private rings matter: mbarrier parity waits are only sound if a waiter is never two phases away from the barrier, which a
// ring shared by independently progressing consumer groups cannot guarantee.
constexpr uint32_t U_OFF = LAT_OFF + 2 * LAT_HALF;
#ifndef DESMO_U_ROWS
#define DESMO_U_ROWS 32
#endif
constexpr int U_ROWS = DESMO_U_ROWS;                   // snapshots per TMA stage
constexpr int U_PER = QT / U_ROWS;                     // stages a quarter consumes per slab-tile
#ifndef DESMO_U_RING
#define DESMO_U_RING 1
#endif
constexpr int U_RING = DESMO_U_RING;                   // stages in a quarter's ring
constexpr uint32_t U_STAGE = U_ROWS * BP * 4;          // must be a multiple of 128 B, the TMA destination alignment
template <bool kU16>
constexpr uint32_t u_stage() { return U_ROWS * BP * (kU16 ? 2 : 4); }  // bytes of one stage of U's element type
constexpr uint32_t TRACE_OFF = U_OFF + NQ * U_RING * U_STAGE;  // debug builds only: 6 event logs of TRACE_LEN entries
constexpr int TRACE_LEN = 384;
constexpr uint32_t SMEM_BYTES = TRACE_OFF + 1024;  // + alignment slack
constexpr uint32_t SMEM_BYTES_DEBUG = SMEM_BYTES + 6 * TRACE_LEN * 8;
static_assert(SMEM_BYTES + 2048 <= 232448, "dynamic + static shared memory must fit the 227 KB of an sm_100 CTA");
static_assert(QT % U_ROWS == 0 && u_stage<true>() % 128 == 0 && U_RING >= U_PER, "U stage shape");
constexpr uint32_t TMEM_REC = 0, TMEM_D = 128, TMEM_G = 192, TMEM_E = 256;  // D: NPR column blocks of 32 (N-stacked B planes), summed in the epilogue
// G1's A operand (the three bf16 planes of the library tile, [point = lane][lib pair = column], 16 columns per plane) lives in
// TMEM: an SS-mode MMA re-reads its 4 KB A tile from shared memory for every instruction, and shared-memory bandwidth is what
// binds this kernel (ncu: tensor-core operand reads + LSU ~ 80-96 % of the data pipe).
}  // namespace tc

struct TcArgs {
    const void* U;
    const float* P;
    const float* phi;
    const float* omega;
    float* dphi;
    float* Epart;
    double* Spart;
    float* Dacc;   // [Kp][ld] raw dG = R W^T rows (unscaled), consumed by the chain-rule kernel
    long long n, ld;
    int m, mld, r, T, K, nslab, kp_out;
    unsigned long long* dbg;  // optional per-CTA phase timers (cycles), 32 per CTA
    float scale;
    uint32_t zero;     // always 0, but only the host knows: lets an address depend on a value without changing it (U-stage release)
    float seed_scale;  // kSupplied: factor applied to the supplied upstream gradient (n_global * m / 2, undoing the MSE scale downstream)
    MonoTable mt;
};

// ------------------------------------------------------------------------------------------------- PTX helpers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint32_t sw128(uint32_t row, uint32_t byte_in_row) {
    return row * 128u + ((((byte_in_row >> 4) ^ (row & 7u)) << 4) | (byte_in_row & 15u));
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ unsigned long long* g_tc_dbg = nullptr;  // host-mapped diagnostics buffer (DESMO_TC_DEBUG), survives a trap
template <bool kDebug>
__device__ __forceinline__ void mbar_wait_t(uint32_t bar, uint32_t parity, int tag, int iter) {
    uint32_t done = 0;
    unsigned spins = 0;
    while (!done) {
        // the suspend-time hint lets the hardware park the thread instead of burning issue slots the epilogue math needs
        asm volatile("{\n\t.reg .pred q;\n\tmbarrier.try_wait.parity.shared::cta.b64 q, [%1], %2, %3;\n\tselp.u32 %0, 1, 0, q;\n\t}\n"
                     : "=r"(done) : "r"(bar), "r"(parity), "r"(kDebug ? 2000u : 0x989680u) : "memory");
        if (kDebug && !done && ++spins >= (1u << 20)) {
            // debug runs report who was stuck where (production runs rely on the CTA's watchdog lane: a spin counter in every
            // wait loop was measured to cost 6 % of the kernel)
            if (spins == (1u << 20) && g_tc_dbg) {
                unsigned long long* d = g_tc_dbg + 4096 + (blockIdx.x * 20 + (threadIdx.x >> 5)) * 4;
                d[0] = 0xdead0000ull | (unsigned)tag; d[1] = (unsigned long long)iter; d[2] = parity; d[3] = threadIdx.x;
                __threadfence_system();
            }
            if (spins > (1u << 22)) __trap();
        }
    }
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                 ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(bar) : "memory");
}
// One non-blocking test of a phase, without a retry loop.  A SYNCS round trip costs a few hundred cycles under this kernel's
// shared-memory load even when the phase completed long ago; a straight-line probe lets ptxas place independent work (or a second
// probe) under that latency, which a wait loop (a branch after every attempt) cannot.  test_wait, not try_wait: try_wait may park the
// warp for a system-dependent time when the phase is still open, which would stall exactly the work the probe is meant to overlap
// (seen in the two-group experiment, profiles/README.md).  Callers fall back to mbar_wait when the probe fails.
__device__ __forceinline__ uint32_t mbar_probe(uint32_t bar, uint32_t parity) {
    uint32_t done;
    asm volatile("{\n\t.reg .pred q;\n\tmbarrier.test_wait.parity.shared::cta.b64 q, [%1], %2;\n\tselp.u32 %0, 1, 0, q;\n\t}\n"
                 : "=r"(done) : "r"(bar), "r"(parity) : "memory");
    return done;
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    return (uint64_t)((saddr >> 4) & 0x3fff) | ((uint64_t)((lbo_bytes >> 4) & 0x3fff) << 16) |
           ((uint64_t)((sbo_bytes >> 4) & 0x3fff) << 32) | ((uint64_t)1 << 46) | ((uint64_t)2 << 61);  // version 1, SWIZZLE_128B
}
__device__ __forceinline__ constexpr uint32_t make_idesc_bf16(int M, int N, int a_mn, int b_mn) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)a_mn << 15) | ((uint32_t)b_mn << 16) | ((uint32_t)(N >> 3) << 17) |
           ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void mma_bf16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
        ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// Collector hints: consecutive MMAs that read the SAME A tile (or, for the weight-stationary form, the same B tile) keep it in the
// tensor core's operand collector instead of fetching it from shared memory again -- shared-memory bandwidth binds this kernel.
// mode: 0 = plain, 1 = fill (read and keep), 2 = use (reuse and keep), 3 = lastuse (reuse and release)
template <int kMode>
__device__ __forceinline__ void mma_bf16_ca(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    if (kMode == 1)
        asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                     "tcgen05.mma.cta_group::1.kind::f16.collector::a::fill [%0], %1, %2, %3, p;\n\t}\n"
                     ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
    else if (kMode == 2)
        asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                     "tcgen05.mma.cta_group::1.kind::f16.collector::a::use [%0], %1, %2, %3, p;\n\t}\n"
                     ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
    else if (kMode == 3)
        asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                     "tcgen05.mma.cta_group::1.kind::f16.collector::a::lastuse [%0], %1, %2, %3, p;\n\t}\n"
                     ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
    else
        mma_bf16(d_tmem, adesc, bdesc, idesc, accumulate);
}
// weight-stationary form, A in tensor memory, B from shared memory through collector buffer b0
template <int kMode>
__device__ __forceinline__ void mma_bf16_ts_wsb(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    if (kMode == 1)
        asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                     "tcgen05.mma.ws.cta_group::1.kind::f16.collector::b0::fill [%0], [%1], %2, %3, p;\n\t}\n"
                     ::"r"(d_tmem), "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
    else if (kMode == 2)
        asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                     "tcgen05.mma.ws.cta_group::1.kind::f16.collector::b0::use [%0], [%1], %2, %3, p;\n\t}\n"
                     ::"r"(d_tmem), "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
    else if (kMode == 3)
        asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                     "tcgen05.mma.ws.cta_group::1.kind::f16.collector::b0::lastuse [%0], [%1], %2, %3, p;\n\t}\n"
                     ::"r"(d_tmem), "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
    else
        asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                     "tcgen05.mma.ws.cta_group::1.kind::f16.collector::b0::discard [%0], [%1], %2, %3, p;\n\t}\n"
                     ::"r"(d_tmem), "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t* v) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
                   "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
                 : "r"(taddr) : "memory");
}
__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ void st_shared_u16(uint32_t addr, uint16_t v) {
    asm volatile("st.shared.u16 [%0], %1;" ::"r"(addr), "h"(v) : "memory");
}
__device__ __forceinline__ bool elect_one_sync() {
    uint32_t pred = 0;
    asm volatile("{\n\t.reg .b32 rx;\n\t.reg .pred px;\n\telect.sync rx|px, %1;\n\t@px mov.s32 %0, 1;\n\t}\n" : "+r"(pred) : "r"(0xffffffffu));
    return pred != 0;
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t* v) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]) : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_st1(uint32_t taddr, uint32_t v) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x1.b32 [%0], {%1};" ::"r"(taddr), "r"(v) : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// A operand in tensor memory (128 lanes = rows, 8 columns = 16 bf16 along K), B from shared memory
__device__ __forceinline__ void mma_bf16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}\n"
        ::"r"(d_tmem), "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}

// x ~ b1 + b2 (bf16 each, round-to-nearest): packs two consecutive elements (lo = first) per 32-bit word
// (the conversions are `volatile` so that the compiler cannot sink them below the mbarrier wait that follows them in the epilogue)
__device__ __forceinline__ void split2_pair(float x0, float x1, uint32_t& w1, uint32_t& w2) {
    asm volatile("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(w1) : "f"(x1), "f"(x0));
    const float e0 = x0 - __uint_as_float(w1 << 16), e1 = x1 - __uint_as_float(w1 & 0xffff0000u);
    asm volatile("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(w2) : "f"(e1), "f"(e0));
}

// The six (a-plane, b-plane) products kept by the 3-way split (i + j <= 4), smallest contributions first.
// Descriptors: the high word is constant per operand role; the low word is (addr >> 4) | (LBO >> 4) << 16, so stepping through
// planes / k-steps is ONE 32-bit add of a compile-time constant per operand (smem addresses < 256 KB never carry out of 14 bits).
#define DESMO_PAIRS(X) X(2, 0) X(0, 2) X(1, 1) X(1, 0) X(0, 1) X(0, 0)
#define DESMO_GRAD_PAIRS(X) X(1, 0) X(0, 1) X(0, 0)
__device__ __forceinline__ uint64_t desc_from(uint32_t lo, uint32_t hi) { return ((uint64_t)hi << 32) | lo; }
constexpr uint32_t kDescHi = (1024u >> 4) | (1u << 14) | (2u << 29);  // SBO = 1024 B, version 1, SWIZZLE_128B

// kSupplied: backward of forward()'s reconstruction for an arbitrary upstream gradient (desmo_recon_backward): the buffer read through
// the U path holds dL/drecon, R := seed_scale * (that) instead of G W - U, G1 is skipped; G3 / G4 / hand-overs are unchanged.
// kU16: U holds bf16 snapshots; the epilogue widens each one exactly to fp32 (a 16-bit shift), all arithmetic after the load is the same.
template <bool kDebug, bool kSupplied, bool kU16>
__global__ void __launch_bounds__(tc::THREADS, 1) fused_tc_kernel(const TcArgs a, const __grid_constant__ CUtensorMap tmW,
                                                                          const __grid_constant__ CUtensorMap tmU,
                                                                          const __grid_constant__ CUtensorMap tmPhi,
                                                                          const __grid_constant__ CUtensorMap tmP) {
    using namespace tc;
    static_assert(!(kSupplied && kU16), "recon_backward reads an fp32 upstream gradient");
    constexpr uint32_t US = u_stage<kU16>();  // bytes per U stage
    constexpr uint32_t UB = kU16 ? 2 : 4;     // bytes per snapshot element
    extern __shared__ uint8_t smem_raw[];
    enum { W_FULL0 = 0, W_FULL1, W_EMPTY0, W_EMPTY1, REC_FULL, REC_EMPTY, R_FULL, GT_FULL, LAT_FULL, LAT_EMPTY, D_FULL, D_EMPTY,
           R_EMPTYQ0, U_FULL0 = R_EMPTYQ0 + 4, U_EMPTY0 = U_FULL0 + NQ * U_RING, NBARS = U_EMPTY0 + NQ * U_RING };
    __shared__ __align__(8) uint64_t bars[NBARS];
    __shared__ uint32_t tmem_base_s;
    __shared__ uint32_t sink_s[32];  // write-only (see the epilogue)
    __shared__ float omega_s[3 * kMaxR];
    __shared__ uint32_t desc_s[KP];  // packed description of library term j: kind | deg << 3 | mode indices (3 bits each) << 6
    __shared__ double red_s[4];
    __shared__ volatile int progress_s;  // slab-tiles the MMA issuer has completed issuing (watchdog)
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    const uint32_t sbase = smem_u32(smem);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (kDebug) for (int i = tid; i < 6 * TRACE_LEN; i += THREADS) reinterpret_cast<unsigned long long*>(smem + TRACE_OFF)[i] = 0ull;
    auto bar = [&](int i) { return smem_u32(&bars[i]); };
    auto mbar_wait = [&](uint32_t b, uint32_t parity, int tag = 0, int iter = 0) { mbar_wait_t<kDebug>(b, parity, tag, iter); };
    auto now = [&]() -> long long { return kDebug ? clock64() : 0ll; };
    // debug timeline of CTA 0 (tools/tc_timeline.py): per-role logs of (tag, iteration, clock) for a window of slab-tiles
    // (kept in shared memory behind the U rings and copied out at the end: a store to mapped host memory per event would stall the roles)
    int trc = 0;
    unsigned long long* trace_s = reinterpret_cast<unsigned long long*>(smem + TRACE_OFF);
    auto trace = [&](int log, int tag, int it_) {
        if (kDebug && blockIdx.x == 0 && a.dbg && it_ >= 24 && it_ < 48 && trc < TRACE_LEN)
            trace_s[log * TRACE_LEN + trc++] = ((unsigned long long)tag << 56) | ((unsigned long long)it_ << 40) | (clock64() & 0xffffffffffull);
    };

    const int nslab = a.nslab;
    const long long ntiles = a.ld / BP;
    const int my_tiles = (int)((ntiles - blockIdx.x + gridDim.x - 1) / gridDim.x);
    const int total = my_tiles * nslab;

    if (tid == 32) {
        mbar_init(bar(W_FULL0), 1); mbar_init(bar(W_FULL1), 1); mbar_init(bar(W_EMPTY0), 1); mbar_init(bar(W_EMPTY1), 1);
        mbar_init(bar(REC_FULL), 1); mbar_init(bar(REC_EMPTY), EPI_THREADS); mbar_init(bar(R_FULL), EPI_THREADS);
        mbar_init(bar(GT_FULL), EPI_THREADS); mbar_init(bar(LAT_FULL), 1); mbar_init(bar(LAT_EMPTY), EPI_THREADS);
        mbar_init(bar(D_FULL), 1); mbar_init(bar(D_EMPTY), EPI_THREADS);
        for (int i = 0; i < NQ * U_RING; ++i) { mbar_init(bar(U_FULL0 + i), 1); mbar_init(bar(U_EMPTY0 + i), 128); }
        for (int i = 0; i < 4; ++i) mbar_init(bar(R_EMPTYQ0 + i), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (tid < 4) red_s[tid] = 0.0;
    if (tid == 0) progress_s = 0;
    if (tid < 3 * a.r) omega_s[tid] = a.omega[tid];
    if (tid >= 64 && tid < 64 + KP) {
        // term j of the library (CYL:376-434 column order, then the sin / cos / tanh blocks of CYL:565-567)
        const int j = tid - 64;
        uint32_t d = 4u;  // padding column: identically zero
        if (j < a.T) {
            const int deg = a.mt.deg[j];
            d = (uint32_t)deg << 3;
            for (int q = 0; q < deg; ++q) d |= (uint32_t)a.mt.idx[j][q] << (6 + 3 * q);
        } else if (j < a.K) {
            const int b = (j - a.T) / a.r, i = (j - a.T) - b * a.r;
            d = (uint32_t)(1 + b) | ((uint32_t)i << 6);
        }
        desc_s[j] = d;
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_base_s;

    // Register budget (setmaxnreg, per warpgroup of four warps): the control warpgroup keeps 32 registers per thread and hands the rest
    // of its launch-time allocation to the four epilogue warpgroups -- 128 * 32 + 512 * 112 = 640 * 96.  With 112 registers the
    // epilogue keeps its addresses and loop invariants resident instead of rematerialising them every slab (and nothing spills).
    if (warp < 4) {
#if DESMO_SETMAXNREG
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(REGS_CTRL));
#endif
    if (warp == 0) {
        // ======================== TMA producer: W slab planes; phi / P rows of the tile whose library is evaluated next ========================
        if (elect_one_sync()) {
            asm volatile("prefetch.tensormap [%0];" ::"l"(&tmW) : "memory");
            for (int it = 0; it < total; ++it) {
                const int buf = it & 1, slab = it % nslab;
                if (it >= 2) mbar_wait(bar(W_EMPTY0 + buf), ((it >> 1) & 1) ^ 1, 1, it);
                mbar_expect_tx(bar(W_FULL0 + buf), W_SLAB);
                for (int h = 0; h < 2; ++h)
                    tma_load_2d(sbase + W_OFF + buf * W_SLAB + h * W_BOX, &tmW, slab * BT + h * 64, 0, bar(W_FULL0 + buf));
            }
        } else if (lane == 3) {
            // phi / P rows of the tile whose library is evaluated next: one buffer, refilled as soon as the epilogue has released it
            // (LAT_EMPTY).  A lane of its own: the W loop above blocks on W_EMPTY, which (with one slab per tile) the MMA issuer
            // only commits after the next tile's first G1 -- which needs these rows.  Found by the watchdog on a 40000 x 100 case.
            asm volatile("prefetch.tensormap [%0];" ::"l"(&tmPhi) : "memory");
            asm volatile("prefetch.tensormap [%0];" ::"l"(&tmP) : "memory");
            for (int k = 0; k < my_tiles; ++k) {
                if (k > 0) mbar_wait(bar(LAT_EMPTY), (k - 1) & 1, 13, k);
                const int x0 = (int)((blockIdx.x + (long long)k * gridDim.x) * BP);
                mbar_expect_tx(bar(LAT_FULL), 2u * a.r * BP * 4u);
                tma_load_2d(sbase + LAT_OFF, &tmPhi, x0, 0, bar(LAT_FULL));
                tma_load_2d(sbase + LAT_OFF + LAT_HALF, &tmP, x0, 0, bar(LAT_FULL));
            }
        } else if (lane == 2) {
            // Watchdog: a protocol error must fail the launch, not hang the GPU.  One otherwise idle lane naps and checks that the
            // MMA issuer keeps advancing; ~2 s without progress traps.  Short naps: the CTA cannot retire before this lane has seen
            // the last slab-tile issued (a 20 us nap cost the script-sized shapes 10-20 us per launch).
            int last = -1;
            unsigned idle = 0;
            for (;;) {
                const int pr = progress_s;
                if (pr >= total) break;
                if (pr != last) { last = pr; idle = 0; }
                else if (++idle > 2000000u) __trap();
                __nanosleep(1000);
            }
        } else if (kDebug && lane == 1 && blockIdx.x == 0) {
            // debug timeline: when the tensor pipe's commits actually land (polled in issue order: G1(it), then G4(it - 1))
            for (int it = 0; it < total && it < 48; ++it) {
                mbar_wait(bar(REC_FULL), it & 1, 15, it);
                trace(5, 50, it);
                if (it > 0) { mbar_wait(bar(R_EMPTYQ0 + 3), (it - 1) & 1, 16, it); trace(5, 51, it - 1); }
            }
        }
    } else if (warp == 3 || warp == 2) {
        // ================= TMA producers: U boxes [U_ROWS snapshots][128 points]; each thread feeds the private rings of two quarters ======
        // A quarter consumes U_PER stages per slab-tile; the box of a stage is requested as soon as the stage's previous contents are
        // consumed.  No divisions in the loop: one thread sustains ~1 TMA instruction per 400 cycles.  (Pulling the next slab-tile
        // into L2 ahead of the ring -- by TMA prefetches or by plain prefetch instructions of the idle lanes -- was measured
        // 9-18 % SLOWER, profiles/README.md: the rings are not what this kernel waits for.)
        if (elect_one_sync()) {
            asm volatile("prefetch.tensormap [%0];" ::"l"(&tmU) : "memory");
            const int h0 = (warp - 2) * 2;
            int slab = 0, st = 0, use = 0;  // ring position and how often the ring has wrapped
            long long tile = blockIdx.x;
            unsigned long long tp0 = 0;
            const long long tps = now();
            for (int it = 0; it < total; ++it) {
#pragma unroll
                for (int k = 0; k < U_PER; ++k) {
#pragma unroll
                    for (int hh = 0; hh < 2; ++hh) {
                        const int b = (h0 + hh) * U_RING + st;
                        long long cp0 = now();
                        if (use > 0) mbar_wait(bar(U_EMPTY0 + b), (use - 1) & 1, 2, it);
                        tp0 += now() - cp0;
#ifdef EXP_NO_UTMA
                        mbar_arrive(bar(U_FULL0 + b));
#else
                        mbar_expect_tx(bar(U_FULL0 + b), US);
                        tma_load_2d(sbase + U_OFF + b * US, &tmU, (int)(tile * BP), slab * BT + (h0 + hh) * QT + k * U_ROWS, bar(U_FULL0 + b));
#endif
                    }
                    if (++st == U_RING) { st = 0; ++use; }
                }
                if (++slab == nslab) { slab = 0; tile += gridDim.x; }
            }
            if (a.dbg) { a.dbg[blockIdx.x * 32 + 20 + (warp - 2) * 2] = tp0; a.dbg[blockIdx.x * 32 + 21 + (warp - 2) * 2] = now() - tps; }
        }
    } else if (warp == 1) {
        // ================================================ MMA issuer ================================================
        if (elect_one_sync()) {
            constexpr uint32_t idesc_g1 = make_idesc_bf16(BP, BT, 0, 1);  // A from TMEM: rows = lanes, K along columns; B = W_s MN-major
            constexpr uint32_t idesc_g4 = make_idesc_bf16(BT, KP, 1, 0);
            unsigned long long tm[6] = {0, 0, 0, 0, 0, 0};
            auto issue_g1 = [&](int it) {
                const int buf = it & 1, slab = it % nslab, tl = it / nslab;
                long long c0 = now();
                trace(0, 1, it);
                mbar_wait(bar(W_FULL0 + buf), (it >> 1) & 1, 3, it);
                long long c1 = now(); tm[0] += c1 - c0;
                trace(0, 2, it);
                if (it > 0) mbar_wait(bar(REC_EMPTY), (it - 1) & 1, 4, it);
                c0 = now(); tm[1] += c0 - c1;
                trace(0, 3, it);
                if (slab == 0) mbar_wait(bar(GT_FULL), tl & 1, 5, it);
                c1 = now(); tm[2] += c1 - c0;
                trace(0, 4, it);
                tc_fence_after();
                // A = library planes in TMEM (16 columns per plane, 8 per k-step), B = W_s MN-major (N = snapshots, 2 boxes LBO = W_BOX)
                const uint32_t wa_lo = ((sbase + W_OFF + buf * W_SLAB) >> 4) | ((W_BOX >> 4) << 16);
                uint32_t acc = 0;
#if DESMO_G1_WS
                // weight-stationary form: the W tile of a (plane, k-step) stays in the collector for all library planes it multiplies
#define G1_WS(PA, PB, MODE)                                                                                          \
    mma_bf16_ts_wsb<MODE>(tmem + TMEM_REC, tmem + TMEM_G + PA * (KP / 2) + ks * 8,                                    \
                          desc_from(wa_lo + ((PB * W_PLANE + ks * 2048) >> 4), kDescHi), idesc_g1, acc);               \
    acc = 1;
#ifndef EXP_NO_G1
                if (!kSupplied) {
#pragma unroll
                    for (int ks = 0; ks < KP / 16; ++ks) { G1_WS(0, 2, 0) G1_WS(1, 1, 1) G1_WS(0, 1, 3) G1_WS(2, 0, 1) G1_WS(1, 0, 2) G1_WS(0, 0, 3) }
                }
#endif
#undef G1_WS
#else
#define G1_PAIR(PA, PB)                                                                                              \
    _Pragma("unroll") for (int ks = 0; ks < KP / 16; ++ks) {                                                          \
        mma_bf16_ts(tmem + TMEM_REC, tmem + TMEM_G + PA * (KP / 2) + ks * 8,                                          \
                    desc_from(wa_lo + ((PB * W_PLANE + ks * 2048) >> 4), kDescHi), idesc_g1, acc);                     \
        acc = 1;                                                                                                      \
    }
#ifndef EXP_NO_G1
                if (!kSupplied) { DESMO_PAIRS(G1_PAIR) }
#endif
#undef G1_PAIR
#endif
                umma_commit(bar(REC_FULL));
                trace(0, 5, it);
            };
            auto issue_g34 = [&](int it) {
                const int buf = it & 1, slab = it % nslab, tl = it / nslab;
                long long c0 = now();
                trace(0, 6, it);
                mbar_wait(bar(R_FULL), it & 1, 6, it);
                long long c1 = now(); tm[3] += c1 - c0;
                trace(0, 7, it);
                if (slab == 0 && tl > 0) mbar_wait(bar(D_EMPTY), (tl - 1) & 1, 7, it);
                c0 = now(); tm[4] += c0 - c1;
                tc_fence_after();
                const uint32_t rk_lo = ((sbase + R_OFF) >> 4) | (1u << 16);                       // R_s K-major (G3 A)
                const uint32_t rm_lo = ((sbase + R_OFF) >> 4) | ((BP * 128u >> 4) << 16);         // R_s MN-major (G4 A), LBO = 16384
                const uint32_t wk_lo = ((sbase + W_OFF + buf * W_SLAB) >> 4) | (1u << 16);        // W_s K-major (G3 B)
                const uint32_t gk_lo = ((sbase + G_OFF) >> 4) | (1u << 16);                       // G_s K-major (G4 B)
                // G3: D += R W^T   (K = snapshots: 8 k-steps of 16; box = ks / 4, 32 B per k-step inside the swizzled row).
                // The B planes are stacked along N: plane a of R multiplies planes 0..1-a of W in ONE MMA of N = 32*(2-a); column
                // block b of D then holds sum_a R_a W_b and the blocks are added when D is read (A is fetched 2x, not 3x).
                uint32_t acc0 = slab > 0 ? 1u : 0u;
#define G3_PLANE(PA)                                                                                                 \
    _Pragma("unroll") for (int ks = 0; ks < BT / 16; ++ks) {                                                          \
        mma_bf16(tmem + TMEM_D, desc_from(rk_lo + ((PA * R_PLANE + (ks >> 2) * (BP * 128) + (ks & 3) * 32) >> 4), kDescHi), \
                 desc_from(wk_lo + (((ks >> 2) * W_BOX + (ks & 3) * 32) >> 4), kDescHi), make_idesc_bf16(BP, KP * (NPR - PA), 0, 0), \
                 (PA == 0) ? acc0 : 1u);                                                                              \
        if (PA == 0) acc0 = 1;                                                                                        \
    }
#ifndef EXP_NO_G3
                G3_PLANE(0) G3_PLANE(1)
#endif
#undef G3_PLANE
                umma_commit(bar(W_EMPTY0 + buf));  // W slab is dead after G3: let the producer refill it while G4 runs
                trace(0, 9, it);
                uint32_t acc = (tl % E_FLUSH_TILES) > 0 ? 1u : 0u;  // fresh E accumulators after every flush
                const uint32_t e_tmem = tmem + TMEM_E + slab * KP;
                // G4: E^T += R^T G  (K = points: 8 k-steps of 16 rows = 2048 B; B = G_s K-major, box = ks / 4).  Issued lane quadrant
                // by lane quadrant (k-steps 2q, 2q+1 read the R_s rows and G_s columns of points 32q..32q+31 only) with one commit each:
                // the epilogue warps of quadrant q may overwrite their part of R_s (and, at a tile boundary, of G_s) while G4 still
                // works on the later quadrants, so only the LAST quadrant's stores are serialised between G4 of this slab and G3 of the next.
                // The two products of R's first plane read the same A tile back to back: the second takes it from the collector.
#define G4_MMA(PA, PB, MODE)                                                                                         \
    mma_bf16_ca<DESMO_G4_COLLECT ? MODE : 0>(e_tmem, desc_from(rm_lo + ((PA * R_PLANE + ks * 2048) >> 4), kDescHi),    \
        desc_from(gk_lo + ((PB * G_PLANE + (ks >> 2) * (KP * 128) + (ks & 3) * 32) >> 4), kDescHi), idesc_g4, acc);    \
    acc = 1;
#pragma unroll
                for (int qq = 0; qq < 4; ++qq) {
#ifndef EXP_NO_G4
#pragma unroll
                    for (int kk = 0; kk < 2; ++kk) {
                        const int ks = 2 * qq + kk;
                        G4_MMA(1, 0, 0) G4_MMA(0, 1, 1) G4_MMA(0, 0, 3)
                    }
#endif
                    umma_commit(bar(R_EMPTYQ0 + qq));
                    trace(0, 10 + qq, it);
                }
#undef G4_MMA
                if (slab == nslab - 1) umma_commit(bar(D_FULL));
            };
            if (total > 0) issue_g1(0);
            for (int it = 0; it < total; ++it) {
                // run ahead, across tile boundaries too: the tensor pipe works on G1 of the next slab-tile while the epilogue forms R
                if (it + 1 < total) issue_g1(it + 1);
                issue_g34(it);
                progress_s = it + 1;
            }
            if (a.dbg) for (int i = 0; i < 5; ++i) a.dbg[blockIdx.x * 32 + i] = tm[i];
        }
    }
    } else {
#if DESMO_SETMAXNREG
        asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(REGS_EPI));
#endif
        // ================================================ epilogue warps ================================================
        // thread <-> (mesh point p == TMEM lane, quarter h of the slab's snapshots): 16 warps, q = lane quadrant, h = snapshots 32h..32h+31
        const int e = warp - 4, q = e & 3, h = e >> 2;
        const int elog = (lane == 0 && (e == 0 || e == 5 || e == 10 || e == 15)) ? 1 + e / 5 : -1;
        auto etrace = [&](int tag, int it_) { if (kDebug && elog >= 0) trace(elog, tag, it_); };
        const int p = q * 32 + lane;
        const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
        double loss_acc = 0.0;
        unsigned long long te[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        const long long tstart = now();

        auto store_d = [&](int tile_local, long long tile) {
            // D = R W^T of the finished tile: quarter h drains library columns 8h..8h+7 (the N-stacked blocks summed) to Dacc[j][x];
            // the chain rule through POOL_DATA / sin / cos / tanh runs in a separate light kernel, off this kernel's critical path.
            const long long x = tile * BP + p;
            mbar_wait(bar(D_FULL), tile_local & 1, 8, tile_local);
            tc_fence_after();
            uint32_t v0[8], v1[8];
            tmem_ld8(tmem + lane_addr + TMEM_D + h * 8, v0);
            tmem_ld8(tmem + lane_addr + TMEM_D + KP + h * 8, v1);
            tmem_ld_wait();
            if ((tile_local + 1) % E_FLUSH_TILES == 0 || tile_local == my_tiles - 1) {
                // E^T accumulators -> this CTA's fp32 partial (round-to-nearest adds), then the MMA issuer restarts them at zero
                const bool first = tile_local < E_FLUSH_TILES;
                float* Eo = a.Epart + (long long)blockIdx.x * a.kp_out * a.mld;
                for (int slab = h; slab < nslab; slab += NQ) {
                    const int t = slab * BT + p;
#pragma unroll
                    for (int c = 0; c < 2; ++c) {
                        uint32_t v[16];
                        float old[16];
                        float* const dst = Eo + (long long)(c * 16) * a.mld + t;
                        const bool mine = t < a.mld;
                        // all 16 partial sums first: independent L2 loads in flight together (one by one each costs a round trip)
#pragma unroll
                        for (int j = 0; j < 16; ++j)
                            old[j] = (mine && !first && c * 16 + j < a.kp_out) ? __ldcg(dst + (long long)j * a.mld) : 0.0f;
                        tmem_ld16(tmem + lane_addr + TMEM_E + slab * KP + c * 16, v);
                        tmem_ld_wait();
                        if (mine) {
#pragma unroll
                            for (int j = 0; j < 16; ++j)
                                if (c * 16 + j < a.kp_out) __stcg(dst + (long long)j * a.mld, old[j] + __uint_as_float(v[j]));
                        }
                    }
                }
            }
#pragma unroll
            for (int j = 0; j < 8; ++j)
                if (h * 8 + j < a.K)  // rows K..Kp-1 of D belong to zero rows of W: never read by the chain rule
                    a.Dacc[(long long)(h * 8 + j) * a.ld + x] = __uint_as_float(v1[j]) + __uint_as_float(v0[j]);
            // the accumulator is handed back only after the loaded registers were consumed: an experiment that arrived on REC_EMPTY
            // straight after tcgen05.wait::ld (before using the data) produced wrong residuals in a few columns (profiles/README.md)
            tc_fence_before();
            mbar_arrive(bar(D_EMPTY));
        };

        // ---- library row of a point (CYL:538-548,565-567).  The four quarters share the work: quarter h owns the library PAIRS
        //      c = h, h+4, h+8, h+12 (terms 2c, 2c+1) -- a pair is one packed word of the TMEM-resident A operand of G1, and the
        //      interleave spreads the sin / cos / tanh terms (the last 3r of K) over the quarters.  The row of the NEXT tile is
        //      evaluated term by term in the slack after each slab's R_FULL hand-over, from the phi / P rows the producer staged in
        //      shared memory; gv[tile parity][.] keeps the fp32 terms until both operand copies (TMEM, G_s) are written. ----
        const float* phi_s = reinterpret_cast<const float*>(smem + LAT_OFF);
        const float* P_s = reinterpret_cast<const float*>(smem + LAT_OFF + LAT_HALF);
        float gv[2][TPT];
        unsigned long long tl2[2] = {0, 0};
        auto term_of = [&](int jj) { return 2 * (h + (jj >> 1) * NQ) + (jj & 1); };
        auto eval_term = [&](int jj) -> float {
            const uint32_t d = desc_s[term_of(jj)];
            const uint32_t kind = d & 7u;
#ifdef EXP_NO_EVAL
            return 0.25f + (float)kind;
#endif
            if (kind == 4u) return 0.0f;
            if (kind == 0u) {  // monomial: left-to-right product of the latent modes, as CYL:390-431
                const int deg = (d >> 3) & 7;
                float v = 1.0f;
                for (int k = 0; k < deg; ++k) {
                    const int i = (d >> (6 + 3 * k)) & 7;
                    const float f = phi_s[i * BP + p] * P_s[i * BP + p];
                    v = (k == 0) ? f : v * f;
                }
                return v;
            }
            const int i = (d >> 6) & 7;
            const float arg = omega_s[3 * i + (int)kind - 1] * (phi_s[i * BP + p] * P_s[i * BP + p]);
#ifdef EXP_NO_TRIG
            return arg;
#endif
            return (kind == 1u) ? sinf(arg) : (kind == 2u) ? cosf(arg) : tanhf(arg);
        };
        int ev_next = 0;       // terms of the next library row evaluated so far
        int ev_tile = 0;       // CTA-local index of the tile that row belongs to
        auto eval_upto = [&](int upto) {
            if (ev_next >= upto) return;
            const long long ce0 = now();
            if (ev_next == 0) mbar_wait(bar(LAT_FULL), ev_tile & 1, 14, ev_tile);
            const long long ce1 = now();
#pragma unroll 1
            for (; ev_next < upto; ++ev_next) gv[ev_tile & 1][ev_next] = eval_term(ev_next);
            // gv was stored, so the ld.shared of phi_s / P_s have returned: the buffer may be refilled
            if (ev_next == TPT) mbar_arrive(bar(LAT_EMPTY));
            if (kDebug) { tl2[0] += ce1 - ce0; tl2[1] += now() - ce1; }
        };
        auto split_term = [&](float v, uint16_t& b1, uint16_t& b2, uint16_t& b3) {
            const __nv_bfloat16 c1 = __float2bfloat16_rn(v);
            const float e1 = v - __bfloat162float(c1);
            const __nv_bfloat16 c2 = __float2bfloat16_rn(e1);
            const __nv_bfloat16 c3 = __float2bfloat16_rn(e1 - __bfloat162float(c2));
            b1 = __bfloat16_as_ushort(c1); b2 = __bfloat16_as_ushort(c2); b3 = __bfloat16_as_ushort(c3);
        };
        auto store_library_tmem = [&](int par) {  // A of G1: TMEM [p lane][lib pairs], three planes of 16 columns
            uint16_t pl[3][TPT];
#pragma unroll
            for (int jj = 0; jj < TPT; ++jj) split_term(gv[par][jj], pl[0][jj], pl[1][jj], pl[2][jj]);
#pragma unroll
            for (int pa = 0; pa < 3; ++pa)
#pragma unroll
                for (int cc = 0; cc < TPT / 2; ++cc)
                    tmem_st1(tmem + lane_addr + TMEM_G + pa * (KP / 2) + h + cc * NQ, (uint32_t)pl[pa][2 * cc] | ((uint32_t)pl[pa][2 * cc + 1] << 16));
            tmem_st_wait();
            tc_fence_before();
            mbar_arrive(bar(GT_FULL));
        };
        auto store_library_smem = [&](int par) {  // B of G4: G_s[lib rows][p contiguous], two planes (published with R_FULL)
            const uint32_t gs = sbase + G_OFF + (p >> 6) * (KP * 128);
            const uint32_t pb = (p & 63) * 2;
#pragma unroll
            for (int jj = 0; jj < TPT; ++jj) {
                uint16_t b1, b2, b3;
                split_term(gv[par][jj], b1, b2, b3);
                const uint32_t off = sw128(term_of(jj), pb);
                st_shared_u16(gs + off, b1);
                st_shared_u16(gs + G_PLANE + off, b2);
            }
        };

        if (my_tiles > 0) {  // first tile: nothing to overlap with
            eval_upto(TPT);
            store_library_tmem(0);
        }
        // terms per slab so that the next row is complete before the tile's last slab (which publishes it to TMEM)
        const int ev_per = nslab > 1 ? (TPT + nslab - 2) / (nslab - 1) : TPT;
        int it = 0;
        for (int tl = 0; tl < my_tiles; ++tl) {
            const long long tile = blockIdx.x + (long long)tl * gridDim.x;
            const long long x = tile * BP + p;
            const bool xin = x < a.n;
            const bool have_next = tl + 1 < my_tiles;
            ev_next = have_next ? 0 : TPT;
            ev_tile = tl + 1;
            float lsum = 0.0f;  // fp32 over the 256 residuals of a tile, folded into the fp64 accumulator once per tile (FP64 adds are slow)
            for (int slab = 0; slab < nslab; ++slab, ++it) {
                const int t0 = slab * BT + h * QT;
                long long c0 = now();
                etrace(20, it);
                const int ub = (it * U_PER) % U_RING;          // ring position of this slab-tile's first stage
                const uint32_t upar = ((it * U_PER) / U_RING) & 1;
                {
                    // both hand-overs are normally complete by now: probe them together (one round trip instead of two)
                    const uint32_t d_rec = mbar_probe(bar(REC_FULL), it & 1), d_u = mbar_probe(bar(U_FULL0 + h * U_RING + ub), upar);
                    if (!d_rec) mbar_wait(bar(REC_FULL), it & 1, 10, it);
                    if (!d_u) mbar_wait(bar(U_FULL0 + h * U_RING + ub), upar, 11, it);
                }
                long long c1 = now(); te[0] += c1 - c0;
                etrace(21, it);
                tc_fence_after();
                if (slab == nslab - 1 && have_next) {
                    // G1 of this tile's last slab has completed (REC_FULL): the TMEM planes of the library may take the next tile's row,
                    // and the MMA issuer can run the next tile's first G1 ahead of this slab's G3 / G4
                    const long long cg0 = now();
                    eval_upto(TPT);
                    store_library_tmem((tl + 1) & 1);
                    te[6] += now() - cg0;
                    etrace(30, it);
                }
                uint32_t u[QT];  // Rec of this thread's 32 snapshots, then r = Rec - U in place
                if (!kSupplied) {
                    tmem_ld16(tmem + lane_addr + TMEM_REC + h * QT, u);
                    tmem_ld16(tmem + lane_addr + TMEM_REC + h * QT + 16, u + 16);
                }
                etrace(22, it);
                if (!kSupplied) tmem_ld_wait();
                etrace(23, it);
                // masked == false for every interior (tile, slab): no per-element selects in the common path
                auto residual = [&](auto masked) {
#pragma unroll
                    for (int k = 0; k < U_PER; ++k) {
                        const int sk = (it * U_PER + k) % U_RING;
                        const int st = h * U_RING + sk;
                        if (k > 0) mbar_wait(bar(U_FULL0 + st), ((it * U_PER + k) / U_RING) & 1, 11, it);
                        const uint32_t us = sbase + U_OFF + st * US + p * UB;
#pragma unroll
                        for (int j = 0; j < U_ROWS; ++j) {
                            float uv;
#ifdef EXP_NO_ULDS
                            uv = __uint_as_float(us);
#else
                            if constexpr (kU16) {
                                uint32_t hv;
                                asm volatile("ld.shared.u16 %0, [%1];" : "=r"(hv) : "r"(us + j * (BP * UB)));
                                uv = __uint_as_float(hv << 16);
                            } else {
                                asm volatile("ld.shared.f32 %0, [%1];" : "=f"(uv) : "r"(us + j * (BP * 4)));
                            }
#endif
                            float rr = kSupplied ? uv * a.seed_scale : __uint_as_float(u[k * U_ROWS + j]) - uv;
                            if (decltype(masked)::value) rr = (xin && t0 + k * U_ROWS + j < a.m) ? rr : 0.0f;
                            u[k * U_ROWS + j] = __float_as_uint(rr);
                            lsum = fmaf(rr, rr, lsum);
                        }
                        // The stage may only be released once the ld.shared above have RETURNED: an mbarrier arrive is not held
                        // back by loads still in flight, and the refilling TMA was observed to overwrite rows 5-7 of a stage under
                        // shared-memory congestion (profiles/README.md).
#ifdef DESMO_U_RELEASE_ADDR
                        // Variant: the arrive's ADDRESS depends on the running sum of squares (AND with a zero only the host knows);
                        // lsum is a chain through every residual of the stage, so with in-order issue the arrive exists only after
                        // the last load has returned.  2 instructions instead of 17; measured equal (4650 vs 4645 cycles), not default.
                        mbar_arrive(bar(U_EMPTY0 + st) + (__float_as_uint(lsum) & a.zero));
#else
                        {   // a store that consumes all the residuals precedes the arrive in the same in-order pipeline
                            uint32_t xx = 0;
#pragma unroll
                            for (int j = 0; j < U_ROWS; ++j) xx ^= u[k * U_ROWS + j];
                            asm volatile("st.shared.b32 [%0], %1;" ::"r"(smem_u32(&sink_s[lane])), "r"(xx) : "memory");
                        }
                        mbar_arrive(bar(U_EMPTY0 + st));
#endif
                    }
                };
                if (xin && (t0 + QT <= a.m)) residual(std::false_type{}); else residual(std::true_type{});
                tc_fence_before();
                mbar_arrive(bar(REC_EMPTY));
                etrace(24, it);
                // ---- r -> two bf16 planes, formed in REGISTERS while G3/G4 of the previous slab still read R_s: only the 8 vector
                //      stores below sit between "R_s free" and "R_s full", i.e. on the tensor pipe's critical path ----
                // (the probe of R_s' release is issued first, so that its round trip runs under the split)
                const uint32_t d_r = it > 0 ? mbar_probe(bar(R_EMPTYQ0 + q), (it - 1) & 1) : 1u;
                uint32_t w1[16], w2[16];
#pragma unroll
                for (int ee = 0; ee < 16; ++ee) split2_pair(__uint_as_float(u[2 * ee]), __uint_as_float(u[2 * ee + 1]), w1[ee], w2[ee]);
#ifndef EXP_NO_SPLIT_PIN
                {
                    // ptxas sinks pure arithmetic below the wait loop to shorten live ranges, which would put the whole split back on
                    // the critical path: consuming every last-plane word (each depends on the words of the planes before it) in a
                    // store that precedes the wait pins the split where it is written.  8 LOP3 + 1 STS per thread and slab.
                    uint32_t xw = 0;
#pragma unroll
                    for (int ee = 0; ee < 16; ++ee) xw ^= w2[ee];
                    asm volatile("st.shared.b32 [%0], %1;" ::"r"(smem_u32(&sink_s[lane])), "r"(xw) : "memory");
                }
#endif
                c0 = now(); te[1] += c0 - c1;
                etrace(25, it);
                if (!d_r) mbar_wait(bar(R_EMPTYQ0 + q), (it - 1) & 1, 12, it);
                c1 = now(); te[2] += c1 - c0;
                etrace(26, it);
                // row p of box (h >> 1), 16 B chunks (h & 1) * 4 .. +3 (8 snapshots each)
                const uint32_t rs = sbase + R_OFF + (h >> 1) * (BP * 128) + p * 128;
#pragma unroll
                for (int c = 0; c < 4; ++c) {
#ifdef EXP_NO_RSTS
                    if (a.m > 0) break;
#endif
                    const uint32_t off = ((uint32_t)(((h & 1) * 4 + c) ^ (p & 7))) << 4;
                    st_shared_v4(rs + off, w1[4 * c], w1[4 * c + 1], w1[4 * c + 2], w1[4 * c + 3]);
                    st_shared_v4(rs + R_PLANE + off, w2[4 * c], w2[4 * c + 1], w2[4 * c + 2], w2[4 * c + 3]);
                }
                // first slab of a tile: G4 of the previous tile has released this lane quadrant of G_s as well (same commit as R_s)
                if (slab == 0) store_library_smem(tl & 1);
                c0 = now(); te[4] += c0 - c1;
                etrace(27, it);
                fence_async_smem();
                mbar_arrive(bar(R_FULL));
                c1 = now(); te[7] += c1 - c0;
                etrace(28, it);
                // slack until the next Rec: drain D of the previous tile (its G3 chain ended with that tile's last slab; the issuer
                // holds this tile's first G3 until D_EMPTY) and evaluate the next terms of the next tile's library row
                if (slab == 0 && tl > 0) store_d(tl - 1, tile - gridDim.x);
                if (slab + 1 < nslab) eval_upto(min(TPT, (slab + 1) * ev_per));
                te[3] += now() - c1;
                etrace(29, it);
            }
            loss_acc += (double)lsum;
        }
        if (a.dbg && tid == 128) {
            for (int i = 0; i < 8; ++i) a.dbg[blockIdx.x * 32 + 8 + i] = te[i];
            a.dbg[blockIdx.x * 32 + 16] = now() - tstart;
            a.dbg[blockIdx.x * 32 + 24] = tl2[0];
            a.dbg[blockIdx.x * 32 + 25] = tl2[1];
        }
        if (a.dbg && lane == 0 && blockIdx.x == 0)
            for (int i = 0; i < 8; ++i) a.dbg[8192 + e * 8 + i] = te[i];
        // D of the last tile, then the E accumulators of this CTA
        if (my_tiles > 0) store_d(my_tiles - 1, blockIdx.x + (long long)(my_tiles - 1) * gridDim.x);
        loss_acc = warp_sum(loss_acc);
        if (lane == 0) atomicAdd(&red_s[q], loss_acc);
        tc_fence_before();
    }
    __syncthreads();
    if (kDebug && blockIdx.x == 0 && a.dbg)
        for (int i = tid; i < 6 * TRACE_LEN; i += THREADS) a.dbg[8320 + i] = trace_s[i];
    for (int i = tid; i < kScal; i += THREADS)
        a.Spart[(long long)blockIdx.x * kScal + i] = (i == 0) ? (((red_s[0] + red_s[1]) + red_s[2]) + red_s[3]) : 0.0;
    if (warp == 2) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512u) : "memory");
    }
}

// ------------------------------------------------------------------------------------------------- host side
// Kernel timing (DESMO_KERNEL_EVENTS=1).  Eager launches record into a ring of event pairs, so that a caller can launch many steps
// back to back (no host synchronisation in between: a launch after an idle gap runs measurably slower) and read the mean afterwards.
// Launches inside a stream capture record one extra pair as EXTERNAL event nodes of the graph: after a replay it holds the kernel's
// duration inside that replay, i.e. inside the caller's timed region.
constexpr int kEvRing = 64;
static cudaEvent_t g_ev[kEvRing][2];
static cudaEvent_t g_cap_ev[2] = {nullptr, nullptr};
static bool g_ev_made = false, g_cap_recorded = false;
static long long g_ev_n = 0;  // eager launches recorded since the last reset
int fused_event_ms(float* ms) {  // duration of the last eager dominant-kernel launch; synchronises
    if (g_ev_n < 1) return DESMO_ERR_ARG;
    cudaEvent_t* p = g_ev[(g_ev_n - 1) % kEvRing];
    if (cudaEventSynchronize(p[1]) != cudaSuccess) return DESMO_ERR_CUDA;
    return cudaEventElapsedTime(ms, p[0], p[1]) == cudaSuccess ? DESMO_OK : DESMO_ERR_CUDA;
}
int fused_event_mean_ms(float* mean_ms, int* launches, int reset) {  // mean over the (at most kEvRing) eager launches since the last reset
    const long long cnt = g_ev_n < kEvRing ? g_ev_n : kEvRing;
    double sum = 0.0;
    for (long long i = g_ev_n - cnt; i < g_ev_n; ++i) {
        cudaEvent_t* p = g_ev[i % kEvRing];
        float ms = 0.0f;
        if (cudaEventSynchronize(p[1]) != cudaSuccess || cudaEventElapsedTime(&ms, p[0], p[1]) != cudaSuccess) return DESMO_ERR_CUDA;
        sum += ms;
    }
    if (mean_ms) *mean_ms = cnt ? (float)(sum / (double)cnt) : 0.0f;
    if (launches) *launches = (int)cnt;
    if (reset) g_ev_n = 0;
    return DESMO_OK;
}
int fused_event_series_ms(float* out, int capacity, int* count) {  // per-launch durations since the last reset, oldest first
    const long long cnt = g_ev_n < kEvRing ? g_ev_n : kEvRing;
    int k = 0;
    for (long long i = g_ev_n - cnt; i < g_ev_n && k < capacity; ++i, ++k) {
        cudaEvent_t* p = g_ev[i % kEvRing];
        if (cudaEventSynchronize(p[1]) != cudaSuccess || cudaEventElapsedTime(out + k, p[0], p[1]) != cudaSuccess) return DESMO_ERR_CUDA;
    }
    if (count) *count = k;
    return DESMO_OK;
}
int fused_event_graph_ms(float* ms) {  // the dominant kernel inside the last replay of a captured step; synchronises
    if (!g_cap_recorded) return DESMO_ERR_ARG;
    if (cudaEventSynchronize(g_cap_ev[1]) != cudaSuccess) return DESMO_ERR_CUDA;
    return cudaEventElapsedTime(ms, g_cap_ev[0], g_cap_ev[1]) == cudaSuccess ? DESMO_OK : DESMO_ERR_CUDA;
}
void fused_event_record(int which, cudaStream_t st) {
    static const bool on = getenv("DESMO_KERNEL_EVENTS") != nullptr;
    if (!on) return;
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(st, &cap) != cudaSuccess) return;
    if (cap != cudaStreamCaptureStatusNone) {
        // events are created by the first eager launch (no resource creation inside a capture); without one, the graph is left alone
        if (g_ev_made && cudaEventRecordWithFlags(g_cap_ev[which], st, cudaEventRecordExternal) == cudaSuccess && which == 1)
            g_cap_recorded = true;
        return;
    }
    if (!g_ev_made) {
        for (int i = 0; i < kEvRing; ++i) { cudaEventCreate(&g_ev[i][0]); cudaEventCreate(&g_ev[i][1]); }
        cudaEventCreate(&g_cap_ev[0]); cudaEventCreate(&g_cap_ev[1]);
        g_ev_made = true;
    }
    if (which == 0) ++g_ev_n;
    cudaEventRecord(g_ev[(g_ev_n - 1) % kEvRing][which], st);
}

static unsigned long long* g_dbg_host = nullptr;
constexpr size_t kDbgWords = 16384;
int tc_debug_read(uint64_t* out, int count) {
    if (!g_dbg_host) return DESMO_ERR_ARG;
    memcpy(out, g_dbg_host, sizeof(uint64_t) * (count < (int)kDbgWords ? count : (int)kDbgWords));
    return DESMO_OK;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                  CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess && qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}

int fused_tc_supported(const desmo_shape* s, int Kp) {
    return (Kp <= tc::KP && s->r <= kMaxR && s->mld <= tc::MAXSLAB * tc::BT && s->ld % 128 == 0 && s->mld % 8 == 0) ? 1 : 0;
}

void reduce_partials_launch(const float* Epart, int nx, long long ecount, const double* Spart, int nslots, int r, float* red, cudaStream_t st,
                            int what);
int chain_rule_launch(const desmo_shape* s, const MonoTable& mt, int T, int Kp, const float* P, const float* phi, const float* omega, float* dphi,
                      const Workspace& ws, int slot_base, int* nslots, cudaStream_t st);

// phase: 0 = the whole pass; 1 = the dominant kernel + the E part of `red` (final for this rank when it returns); 2 = chain rule + the
// scalar tail of `red` (needs the per-CTA partials phase 1 left in the workspace).
template <bool kDebug, bool kSupplied, bool kU16>
static int launch_tc(int grid, uint32_t smem, const TcArgs& a, const CUtensorMap& tm, const CUtensorMap& tmu, const CUtensorMap& tmphi,
                     const CUtensorMap& tmp, cudaStream_t st) {
    DESMO_CUDA(cudaFuncSetAttribute(fused_tc_kernel<kDebug, kSupplied, kU16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    fused_tc_kernel<kDebug, kSupplied, kU16><<<grid, tc::THREADS, smem, st>>>(a, tm, tmu, tmphi, tmp);
    return DESMO_OK;
}

int fused_tc(const desmo_shape* s, const MonoTable& mt, int T, int Kp, const void* U, int u_dtype, const float* P, const float* phi,
             const float* omega, const float* W, float* dphi, float* red, const Workspace& ws, cudaStream_t st, bool supplied, int phase) {
    (void)W;
    if (!fused_tc_supported(s, Kp)) { set_error("tcgen05 path: unsupported shape"); return DESMO_ERR_UNSUPPORTED; }
    if (phase == 2) {
        int dev2 = 0, sms2 = 0;
        DESMO_CUDA(cudaGetDevice(&dev2));
        DESMO_CUDA(cudaDeviceGetAttribute(&sms2, cudaDevAttrMultiProcessorCount, dev2));
        const long long ntiles2 = s->ld / tc::BP;
        const int grid2 = (int)(ntiles2 < sms2 ? ntiles2 : sms2);
        int nchain2 = 0;
        int rc2 = chain_rule_launch(s, mt, T, Kp, P, phi, omega, dphi, ws, grid2, &nchain2, st);
        if (rc2) return rc2;
        reduce_partials_launch(ws.Epart, grid2, (long long)Kp * s->mld, ws.Spart, grid2 + nchain2, s->r, red, st, 2);
        DESMO_CUDA(cudaGetLastError());
        return DESMO_OK;
    }
    EncodeTiledFn enc = encode_fn();
    if (!enc) { set_error("cuTensorMapEncodeTiled not available"); return DESMO_ERR_CUDA; }
    int dev = 0, sms = 0;
    DESMO_CUDA(cudaGetDevice(&dev));
    DESMO_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    // bf16 planes of W written by build_w: Wb[3][Kp_tc][mld]
    CUtensorMap tm;
    const cuuint64_t dims[2] = {(cuuint64_t)s->mld, (cuuint64_t)(3 * tc::KP)};
    const cuuint64_t strides[1] = {(cuuint64_t)s->mld * 2};
    const cuuint32_t box[2] = {64, (cuuint32_t)(3 * tc::KP)};  // one box = all three planes of 64 snapshots
    const cuuint32_t estr[2] = {1, 1};
    CUresult cr = enc(&tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, (void*)ws.tc, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                      CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (cr != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed (%d)", (int)cr); return DESMO_ERR_CUDA; }
    const bool u16 = u_dtype == DESMO_DTYPE_BF16;
    if (u16 && supplied) { set_error("tcgen05 path: recon_backward takes an fp32 upstream gradient"); return DESMO_ERR_ARG; }
    CUtensorMap tmu;
    {
        const cuuint64_t udims[2] = {(cuuint64_t)s->ld, (cuuint64_t)s->m};
        const cuuint64_t ustr[1] = {(cuuint64_t)s->ld * (u16 ? 2 : 4)};
        const cuuint32_t ubox[2] = {(cuuint32_t)tc::BP, (cuuint32_t)tc::U_ROWS};
        cr = enc(&tmu, u16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)U, udims, ustr, ubox, estr,
                 CU_TENSOR_MAP_INTERLEAVE_NONE,
                 CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (cr != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled(U) failed (%d)", (int)cr); return DESMO_ERR_CUDA; }
    }
    CUtensorMap tmphi, tmp;  // rows of phi / P of one tile: box [r][128 points]
    for (int which = 0; which < 2; ++which) {
        const cuuint64_t ldims[2] = {(cuuint64_t)s->ld, (cuuint64_t)s->r};
        const cuuint64_t lstr[1] = {(cuuint64_t)s->ld * 4};
        const cuuint32_t lbox[2] = {(cuuint32_t)tc::BP, (cuuint32_t)s->r};
        cr = enc(which ? &tmp : &tmphi, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)(which ? P : phi), ldims, lstr, lbox, estr,
                 CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (cr != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled(phi / P) failed (%d)", (int)cr); return DESMO_ERR_CUDA; }
    }
    TcArgs a{};
    a.U = U; a.P = P; a.phi = phi; a.omega = omega; a.dphi = dphi; a.Epart = ws.Epart; a.Spart = ws.Spart; a.Dacc = ws.Dacc;
    a.n = s->n; a.ld = s->ld; a.m = s->m; a.mld = s->mld; a.r = s->r; a.T = T; a.K = T + 3 * s->r;
    a.nslab = (s->m + tc::BT - 1) / tc::BT;
    a.dbg = nullptr;
    if (getenv("DESMO_TC_DEBUG")) {
        unsigned long long* dev = nullptr;
        if (!g_dbg_host) {
            DESMO_CUDA(cudaHostAlloc(reinterpret_cast<void**>(&g_dbg_host), kDbgWords * 8, cudaHostAllocMapped));
            memset(g_dbg_host, 0, kDbgWords * 8);
        }
        DESMO_CUDA(cudaHostGetDevicePointer(reinterpret_cast<void**>(&dev), g_dbg_host, 0));
        DESMO_CUDA(cudaMemcpyToSymbolAsync(g_tc_dbg, &dev, sizeof(dev), 0, cudaMemcpyHostToDevice, st));
        a.dbg = dev;
    }
    a.kp_out = Kp;
    a.scale = (float)(2.0 / ((double)s->n_global * (double)s->m));
    a.seed_scale = (float)(0.5 * (double)s->n_global * (double)s->m);
    a.zero = 0u;
    a.mt = mt;
    const long long ntiles = s->ld / tc::BP;
    const int grid = (int)(ntiles < sms ? ntiles : sms);
    fused_event_record(0, st);
    int lrc;
    if (supplied) lrc = launch_tc<false, true, false>(grid, tc::SMEM_BYTES, a, tm, tmu, tmphi, tmp, st);
    else if (a.dbg) lrc = u16 ? launch_tc<true, false, true>(grid, tc::SMEM_BYTES_DEBUG, a, tm, tmu, tmphi, tmp, st)
                              : launch_tc<true, false, false>(grid, tc::SMEM_BYTES_DEBUG, a, tm, tmu, tmphi, tmp, st);
    else lrc = u16 ? launch_tc<false, false, true>(grid, tc::SMEM_BYTES, a, tm, tmu, tmphi, tmp, st)
                   : launch_tc<false, false, false>(grid, tc::SMEM_BYTES, a, tm, tmu, tmphi, tmp, st);
    if (lrc) return lrc;
    fused_event_record(1, st);
    DESMO_CUDA(cudaGetLastError());
    if (phase == 1) {
        reduce_partials_launch(ws.Epart, grid, (long long)Kp * s->mld, ws.Spart, grid, s->r, red, st, 1);
        DESMO_CUDA(cudaGetLastError());
        return DESMO_OK;
    }
    int nchain = 0;
    int rc = chain_rule_launch(s, mt, T, Kp, P, phi, omega, dphi, ws, grid, &nchain, st);
    if (rc) return rc;
    reduce_partials_launch(ws.Epart, grid, (long long)Kp * s->mld, ws.Spart, grid + nchain, s->r, red, st, 3);
    DESMO_CUDA(cudaGetLastError());
    return DESMO_OK;
}

}  // namespace desmo
