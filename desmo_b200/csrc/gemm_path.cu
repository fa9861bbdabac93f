// General-library path (DESMO_PATH_GEMM): libraries beyond what the fused kernel keeps on chip (K > 32 library terms, r up to 64 modes,
// any number of snapshots), e.g. BASELINE's "8 modes" (r = 8, p = 2: K = 69; p = 3: K = 189) and "32 modes" (r = 32, p = 2: K = 657).
//
// With K in the hundreds the three contractions of the step are genuine GEMMs (6 K n m flop on 4 n m bytes: 400 - 1000 flop/B, bound by the
// tensor pipe, not by HBM -- SURVEY.md section 8d), so the step is run as three tcgen05 GEMMs over chunks of mesh points whose residual
// planes stay L2-resident, instead of one fused pass:
//   per chunk of <= 16384 points
//     library_planes_kernel   G = [POOL_DATA(Phi) | sin | cos | tanh]  -> three bf16 planes [3][Kr][chunk]          (CYL:376-434,548,565-567)
//     GEMM 1  Rec = G W       epilogue: r = Rec - U (U read once, fp32), sum r^2, r -> two bf16 planes [2][chunk][mp]   (CYL:572,722)
//     GEMM 3  D   = R W^T     -> Dacc [K][ld] (raw dG, consumed by the chain-rule kernel)
//     GEMM 4  E^T = R^T G     -> per-slice partials of E = G^T R (split over the points of the chunk), accumulated over the chunks
//   chain_rule_generic_kernel (monomial derivatives for any r / p, sin / cos / tanh), gram_phi_kernel (Phi^T Phi), reduce_generic_kernel.
// Precision: every fp32 operand is split into bf16 planes (x = b1 + b2 + b3); Rec keeps the six products with i + j <= 4 (fp32-class: R is a
// small difference), the two gradient GEMMs use two planes / three products (~3e-7 relative, see fused_tc.cu).  The tensor core adds into
// its fp32 accumulators with truncation, so accumulation chains are bounded (kgroup k-blocks per TMEM accumulator, summed in fp32 RN).
//
// One generic kernel, gemm_planes_kernel<A_MN, B_MN, NPA, NPB, EPI>: BM = BN = 128, BK = 64 (one 128 B swizzled row of bf16); warp 0 = TMA
// producer (operand planes through a ring of stages), warp 1 = MMA issuer (one elected thread), warps 2..9 = epilogue (lane quadrant =
// warp % 4, column half = (warp - 2) / 4); two TMEM accumulators (mainloop of the next job overlaps the epilogue of the previous one).
#include <cuda.h>
#include <cuda_bf16.h>
#include <string.h>

#include <type_traits>

#include "common.cuh"
#include "tcgen05.cuh"

namespace desmo {
namespace gp {
using namespace ptx;

constexpr int BM = 128, BN = 128, BK = 64;
constexpr uint32_t PLANE_TILE = 128 * 128;  // bytes of one operand plane tile: 128 rows x 64 bf16 (K-major) or 2 x [64 k-rows x 64 bf16] (MN-major)
constexpr int EPI_WARPS = 8;
constexpr int THREADS = 64 + EPI_WARPS * 32;
constexpr int kChunkPoints = 16384;

// EPI_RESID_BF16: EPI_RESID reading bf16 snapshots.  EPI_PROFILE (_BF16): r = Rec - U as EPI_RESID forms it, reduced to the two marginals of
// r^2 and u^2 (per point, per snapshot) instead of being written out (desmo_residual_profile).
// EPI_PRUNE (_BF16): GEMM 1 transposed (rows = snapshots, columns = points), r = Rec - U as EPI_RESID forms it, then a sequence of
// library terms peeled off one FFMA at a time, reduced to sum_x r_s^2 per snapshot and step (desmo_pruning_profile).
// EPI_GRAM: the residual Gram C_R = R^T R of a chunk (rows and columns = snapshots, contraction over the chunk's points), upper tiles
// only (tn >= tm), per-slice fp64 partials accumulated over the chunks (desmo_residual_gram).
enum { EPI_RESID = 0, EPI_D = 1, EPI_E = 2, EPI_RECON = 3, EPI_RESID_BF16 = 4, EPI_PROFILE = 5, EPI_PROFILE_BF16 = 6, EPI_PRUNE = 7,
       EPI_PRUNE_BF16 = 8, EPI_GRAM = 9 };
// EPI_PROFILE scratch behind the operand stages (dynamic shared memory), two buffers used by alternate tiles:
// [4 lane quadrants][2 column halves][4 blocks of 16 columns][32] per-warp column sums, then [2][128] per-point sums of column half 1
constexpr int kProfSlab = 4 * 2 * 4 * 32 + 2 * 128;
constexpr size_t kProfSmem = 2 * sizeof(float) * kProfSlab;
// EPI_PRUNE scratch behind the operand stages: a of one step chunk [kPruneSteps][BN points], then the fp32 partials of the two column
// halves [2][kPruneSteps + 1][BM snapshots] (row kPruneSteps: sum_x u^2, first chunk only)
constexpr int kPruneSteps = 16;
constexpr size_t kPruneSmem = sizeof(float) * (kPruneSteps * 128 + 2 * (kPruneSteps + 1) * 128);

// ------------------------------------------------------------------------------------------------- PTX helpers (the rest: tcgen05.cuh)
// Every wait carries a watchdog: a protocol error traps (the launch fails with an error) instead of hanging the GPU.
// (Keep this loop's shape: written as while (!mbar_try_wait(...)) it compiles to different register allocations in every GEMM kernel.)
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t done = 0;
    unsigned spins = 0;
    while (!done) {
        done = mbar_try_wait(bar, parity, 20000u);
        if (!done && ++spins > (1u << 18)) __trap();
    }
}
// K-major operand tile [128 rows][128 B]: LBO unused (1); a k-step of 16 elements advances 32 B inside the swizzled row.
// MN-major operand tile, two boxes [64 k-rows][128 B = 64 mn]: LBO = 8192 B (next 64-wide mn block); a k-step of 16 rows advances 2048 B.
template <bool MN>
__device__ __forceinline__ uint64_t operand_desc(uint32_t tile_addr, int ks) {
    if (MN) return desc_from(((tile_addr + ks * 2048) >> 4) | ((8192u >> 4) << 16), kDescHi);
    return desc_from(((tile_addr + ks * 32) >> 4) | (1u << 16), kDescHi);
}
__device__ __forceinline__ void split2_pair(float x0, float x1, uint32_t& w1, uint32_t& w2) {
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(w1) : "f"(x1), "f"(x0));
    const float e0 = x0 - __uint_as_float(w1 << 16), e1 = x1 - __uint_as_float(w1 & 0xffff0000u);
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(w2) : "f"(e1), "f"(e0));
}

// Eight consecutive snapshot values (16-byte aligned) widened exactly to fp32, or zeros when !ok
__device__ __forceinline__ void ldg8_u(const float* p, bool ok, float* u) {
    float4 a = make_float4(0.0f, 0.0f, 0.0f, 0.0f), b = a;
    if (ok) { a = __ldg(reinterpret_cast<const float4*>(p)); b = __ldg(reinterpret_cast<const float4*>(p) + 1); }
    u[0] = a.x; u[1] = a.y; u[2] = a.z; u[3] = a.w; u[4] = b.x; u[5] = b.y; u[6] = b.z; u[7] = b.w;
}
__device__ __forceinline__ void ldg8_u(const __nv_bfloat16* p, bool ok, float* u) {
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    if (ok) v = __ldg(reinterpret_cast<const uint4*>(p));
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) { u[2 * i] = __uint_as_float(w[i] << 16); u[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u); }
}

__device__ __forceinline__ float4 lds_v4(uint32_t addr) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
    return v;
}

struct GemmArgs {
    int tiles_m, tiles_n;      // output tiles (tn fastest in the work order: neighbouring CTAs share the A tile)
    int nslice, kb_per_slice;  // split of the contraction over work items (EPI_E); kb = k-blocks of 64
    int kblocks;               // k-blocks of the whole contraction
    int kgroup;                // k-blocks per TMEM accumulation chain
    int a_rows, b_rows;        // rows per plane of the 2-D maps (planes are stacked along rows)
    int n_lib16;               // valid extent of the library dimension rounded up to 16 (N of the last tile, EPI_D / EPI_E)
    // epilogue
    const void* U;             // EPI_RESID: snapshots [m][ld] fp32 (EPI_RESID_BF16: bf16)
    float* out;                // EPI_RECON: [m][ld]; EPI_PROFILE: per-point partials [tiles_n][2][rows_r] of the chunk
    __nv_bfloat16* Rp;         // EPI_RESID: [2][rows_r][mp]
    float* Dacc;               // EPI_D: [K][ld]
    float* Epart;              // EPI_E: [nslice_alloc][Kp][mld]
    double* loss_part;         // EPI_RESID: [gridDim.x]; EPI_PROFILE: per-CTA snapshot partials [gridDim.x][2][mp], accumulated;
                               // EPI_GRAM: per-slice partials of the upper tiles [nslice][tiles_n][128 t2][128 t1], accumulated
    long long n, ld, x0;       // points of this rank, pitch, first point of the chunk
    long long rows_r;          // rows per plane of Rp (chunk points padded to 128)
    int m, mld, mp, K, Kp;
    int first_chunk;
    // EPI_PRUNE (appended: the fields above keep their offsets): loss_part = per-CTA partials [gridDim.x][steps + 2][BM]
    const float* prune_a;      // [steps + 1][rows_r]: row s = library values of term order[s - 1] at the chunk's points, row 0 = 0
    const float* prune_b;      // [steps + 1][mp]: row s = W[order[s - 1]][t] (0 for t >= m), row 0 = 0
    int steps;
};

// the plane pairs kept by the split, smallest contributions first
template <int NP>
__host__ __device__ constexpr int pair_count() { return NP == 3 ? 6 : 3; }
template <int NP>
__host__ __device__ constexpr int pair_a(int q) {  // 3 planes: (2,0) (0,2) (1,1) (1,0) (0,1) (0,0); 2 planes: (1,0) (0,1) (0,0)
    return NP == 3 ? (q == 0 ? 2 : q == 1 ? 0 : q == 2 ? 1 : q == 3 ? 1 : 0) : (q == 0 ? 1 : 0);
}
template <int NP>
__host__ __device__ constexpr int pair_b(int q) {
    return NP == 3 ? (q == 0 ? 0 : q == 1 ? 2 : q == 2 ? 1 : q == 3 ? 0 : q == 4 ? 1 : 0) : (q == 1 ? 1 : 0);
}

// EPI_GRAM's work items: index i of the upper triangle of a T x T tile grid, row by row -> (tm, tn), tn >= tm
__device__ __forceinline__ int upper_tm(int i, int T) {
    int a = 0;
    while (i >= T - a) { i -= T - a; ++a; }
    return a;
}
__device__ __forceinline__ int upper_tn(int i, int T) {
    const int a = upper_tm(i, T);
    return i - a * T + a * (a - 1) / 2 + a;
}

template <bool A_MN, bool B_MN, int NPA, int NPB, int EPI>
__global__ void __launch_bounds__(THREADS, 1) gemm_planes_kernel(const GemmArgs g, const __grid_constant__ CUtensorMap tmA,
                                                                 const __grid_constant__ CUtensorMap tmB) {
    constexpr uint32_t STAGE = (NPA + NPB) * PLANE_TILE;
    constexpr int NSTAGE = (NPA + NPB) >= 6 ? 2 : 3;
    static_assert(NPA == NPB, "plane pairs are defined for equal plane counts");
    constexpr bool kResid = EPI == EPI_RESID || EPI == EPI_RESID_BF16;
    constexpr bool kProfile = EPI == EPI_PROFILE || EPI == EPI_PROFILE_BF16;
    constexpr bool kPrune = EPI == EPI_PRUNE || EPI == EPI_PRUNE_BF16;
    constexpr bool kGram = EPI == EPI_GRAM;
    using UT = typename std::conditional<EPI == EPI_RESID_BF16 || EPI == EPI_PROFILE_BF16 || EPI == EPI_PRUNE_BF16, __nv_bfloat16, float>::type;
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bars[2 * NSTAGE + 4];
    __shared__ uint32_t tmem_base_s;
    __shared__ double loss_s[EPI_WARPS];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    const uint32_t sbase = smem_u32(smem);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    enum { FULL0 = 0, EMPTY0 = NSTAGE, ACC_FULL0 = 2 * NSTAGE, ACC_EMPTY0 = 2 * NSTAGE + 2 };
    auto bar = [&](int i) { return smem_u32(&bars[i]); };

    if (tid == 32) {
        for (int i = 0; i < NSTAGE; ++i) { mbar_init(bar(FULL0 + i), 1); mbar_init(bar(EMPTY0 + i), 1); }
        for (int i = 0; i < 2; ++i) { mbar_init(bar(ACC_FULL0 + i), 1); mbar_init(bar(ACC_EMPTY0 + i), EPI_WARPS * 32); }
        fence_mbar_init();
    }
    if (warp == 0) tmem_alloc<256>(smem_u32(&tmem_base_s));
    if (tid < EPI_WARPS) loss_s[tid] = 0.0;
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_base_s;

    const int tiles = g.tiles_m * g.tiles_n;
    const int items = tiles * g.nslice;

    if (warp == 0) {
        // ================================================ TMA producer ================================================
        if (elect_one_sync()) {
            asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA) : "memory");
            asm volatile("prefetch.tensormap [%0];" ::"l"(&tmB) : "memory");
            int cnt = 0;
            for (int w = blockIdx.x; w < items; w += gridDim.x) {
                const int slice = w / tiles, rem = w - slice * tiles;
                // EPI_PRUNE: tm fastest -- with gridDim.x a multiple of tiles_m, every tile of a CTA has the same snapshot rows
                const int tm = kGram ? upper_tm(rem, g.mp / BM) : kPrune ? rem % g.tiles_m : rem / g.tiles_n,
                          tn = kGram ? upper_tn(rem, g.mp / BM) : kPrune ? rem / g.tiles_m : rem - tm * g.tiles_n;
                const int kb0 = slice * g.kb_per_slice, kb1 = min(kb0 + g.kb_per_slice, g.kblocks);
                for (int kb = kb0; kb < kb1; ++kb, ++cnt) {
                    const int st = cnt % NSTAGE;
                    if (cnt >= NSTAGE) mbar_wait(bar(EMPTY0 + st), ((cnt / NSTAGE) - 1) & 1);
                    mbar_expect_tx(bar(FULL0 + st), STAGE);
                    const uint32_t sa = sbase + st * STAGE, sb = sa + NPA * PLANE_TILE;
#pragma unroll
                    for (int p = 0; p < NPA; ++p) {
                        if (A_MN) {  // storage [k rows][mn contiguous]: two boxes of 64 mn
                            tma_load_2d(sa + p * PLANE_TILE, &tmA, tm * BM, p * g.a_rows + kb * BK, bar(FULL0 + st));
                            tma_load_2d(sa + p * PLANE_TILE + 8192, &tmA, tm * BM + 64, p * g.a_rows + kb * BK, bar(FULL0 + st));
                        } else {     // storage [mn rows][k contiguous]: one box of 128 rows
                            tma_load_2d(sa + p * PLANE_TILE, &tmA, kb * BK, p * g.a_rows + tm * BM, bar(FULL0 + st));
                        }
                    }
#pragma unroll
                    for (int p = 0; p < NPB; ++p) {
                        if (B_MN) {
                            tma_load_2d(sb + p * PLANE_TILE, &tmB, tn * BN, p * g.b_rows + kb * BK, bar(FULL0 + st));
                            tma_load_2d(sb + p * PLANE_TILE + 8192, &tmB, tn * BN + 64, p * g.b_rows + kb * BK, bar(FULL0 + st));
                        } else {
                            tma_load_2d(sb + p * PLANE_TILE, &tmB, kb * BK, p * g.b_rows + tn * BN, bar(FULL0 + st));
                        }
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ================================================ MMA issuer ================================================
        if (elect_one_sync()) {
            int cnt = 0, job = 0;
            for (int w = blockIdx.x; w < items; w += gridDim.x) {
                const int slice = w / tiles, rem = w - slice * tiles;
                const int tn = rem % g.tiles_n;
                const int kb0 = slice * g.kb_per_slice, kb1 = min(kb0 + g.kb_per_slice, g.kblocks);
                int n_eff = BN;
                if (EPI == EPI_D || EPI == EPI_E) n_eff = min(BN, g.n_lib16 - tn * BN);
                const uint32_t idesc = make_idesc_bf16(BM, n_eff, A_MN ? 1 : 0, B_MN ? 1 : 0);
                for (int kg = kb0; kg < kb1; kg += g.kgroup, ++job) {
                    const int buf = job & 1;
                    if (job >= 2) mbar_wait(bar(ACC_EMPTY0 + buf), ((job >> 1) - 1) & 1);
                    tc_fence_after();
                    const uint32_t acc_tmem = tmem + buf * BN;
                    uint32_t acc = 0;
                    const int kge = min(kg + g.kgroup, kb1);
                    for (int kb = kg; kb < kge; ++kb, ++cnt) {
                        const int st = cnt % NSTAGE;
                        mbar_wait(bar(FULL0 + st), (cnt / NSTAGE) & 1);
                        tc_fence_after();
                        const uint32_t sa = sbase + st * STAGE, sb = sa + NPA * PLANE_TILE;
#pragma unroll
                        for (int q = 0; q < pair_count<NPA>(); ++q) {
#pragma unroll
                            for (int ks = 0; ks < BK / 16; ++ks) {
                                mma_bf16(acc_tmem, operand_desc<A_MN>(sa + pair_a<NPA>(q) * PLANE_TILE, ks),
                                         operand_desc<B_MN>(sb + pair_b<NPA>(q) * PLANE_TILE, ks), idesc, acc);
                                acc = 1;
                            }
                        }
                        umma_commit(bar(EMPTY0 + st));  // stage free once these MMAs have read it
                    }
                    umma_commit(bar(ACC_FULL0 + buf));
                }
            }
        }
    } else {
        // ================================================ epilogue ================================================
        const int q = warp & 3, c = (warp - 2) >> 2;  // TMEM lane quadrant of this warp, column half
        const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
        const int row = q * 32 + lane;  // accumulator row of this thread
        double loss_acc = 0.0;
        int job = 0;
        for (int w = blockIdx.x; w < items; w += gridDim.x) {
            const int slice = w / tiles, rem = w - slice * tiles;
            const int tm = kGram ? upper_tm(rem, g.mp / BM) : kPrune ? rem % g.tiles_m : rem / g.tiles_n,
                      tn = kGram ? upper_tn(rem, g.mp / BM) : kPrune ? rem / g.tiles_m : rem - tm * g.tiles_n;
            const int kb0 = slice * g.kb_per_slice, kb1 = min(kb0 + g.kb_per_slice, g.kblocks);
            float sum[64];
#pragma unroll
            for (int j = 0; j < 64; ++j) sum[j] = 0.0f;
            for (int kg = kb0; kg < kb1; kg += g.kgroup, ++job) {
                const int buf = job & 1;
                mbar_wait(bar(ACC_FULL0 + buf), (job >> 1) & 1);
                tc_fence_after();
#pragma unroll
                for (int blk = 0; blk < 4; ++blk) {
                    uint32_t v[16];
                    tmem_ld16(tmem + lane_addr + buf * BN + c * 64 + blk * 16, v);
                    tmem_ld_wait();
#pragma unroll
                    for (int j = 0; j < 16; ++j) sum[blk * 16 + j] += __uint_as_float(v[j]);  // fp32 round-to-nearest across chains
                }
                tc_fence_before();
                mbar_arrive(bar(ACC_EMPTY0 + buf));
            }
            // ---- finalize the output tile (tm, tn) ----
            const int col0 = tn * BN + c * 64;
            if (kResid) {
                // rows = points of the chunk, columns = snapshots: r = Rec - U, loss, two bf16 planes of r (row-major, t contiguous)
                const long long pl = (long long)tm * BM + row;  // chunk-local point
                const long long x = g.x0 + pl;
                const bool xin = x < g.n;
                float lsum = 0.0f;
#pragma unroll
                for (int blk = 0; blk < 4; ++blk) {
                    float u[16];
#pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        const int t = col0 + blk * 16 + j;
                        u[j] = (xin && t < g.m) ? ldg_u(static_cast<const UT*>(g.U) + (long long)t * g.ld + x) : 0.0f;
                    }
                    uint32_t w1[8], w2[8];
#pragma unroll
                    for (int j = 0; j < 16; j += 2) {
                        const int t = col0 + blk * 16 + j;
                        const float r0 = (xin && t < g.m) ? sum[blk * 16 + j] - u[j] : 0.0f;
                        const float r1 = (xin && t + 1 < g.m) ? sum[blk * 16 + j + 1] - u[j + 1] : 0.0f;
                        lsum = fmaf(r0, r0, lsum);
                        lsum = fmaf(r1, r1, lsum);
                        split2_pair(r0, r1, w1[j >> 1], w2[j >> 1]);
                    }
                    __nv_bfloat16* dst = g.Rp + pl * g.mp + col0 + blk * 16;
                    uint4* d0 = reinterpret_cast<uint4*>(dst);
                    uint4* d1 = reinterpret_cast<uint4*>(dst + g.rows_r * g.mp);
                    d0[0] = make_uint4(w1[0], w1[1], w1[2], w1[3]); d0[1] = make_uint4(w1[4], w1[5], w1[6], w1[7]);
                    d1[0] = make_uint4(w2[0], w2[1], w2[2], w2[3]); d1[1] = make_uint4(w2[4], w2[5], w2[6], w2[7]);
                }
                loss_acc += (double)lsum;
            } else if (EPI == EPI_RECON) {
                const long long x = g.x0 + (long long)tm * BM + row;
#pragma unroll
                for (int j = 0; j < 64; ++j) {
                    const int t = col0 + j;
                    if (t < g.m && x < g.ld) g.out[(long long)t * g.ld + x] = (x < g.n) ? sum[j] : 0.0f;
                }
            } else if (EPI == EPI_D) {
                // rows = points, columns = library terms: raw dG rows, lib-major like the fused kernels' Dacc
                const long long x = g.x0 + (long long)tm * BM + row;
#pragma unroll
                for (int j = 0; j < 64; ++j) {
                    const int k = col0 + j;
                    if (k < g.K && x < g.ld) g.Dacc[(long long)k * g.ld + x] = sum[j];
                }
            } else if (kProfile) {
                // rows = points of the chunk, columns = snapshots: r = Rec - U exactly as EPI_RESID forms it; r^2 and u^2 are summed over
                // this thread's 64 columns (per point) and over the tile's 128 rows (per snapshot), in a fixed order
                const long long pl = (long long)tm * BM + row;  // chunk-local point
                const long long x = g.x0 + pl;
                const bool xin = x < g.n;
                float* prof = reinterpret_cast<float*>(smem + NSTAGE * STAGE) + (((w - (int)blockIdx.x) / (int)gridDim.x) & 1) * kProfSlab;
                float pr = 0.0f, pu = 0.0f;
#pragma unroll
                for (int blk = 0; blk < 4; ++blk) {
                    float u[16];
#pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        const int t = col0 + blk * 16 + j;
                        u[j] = (xin && t < g.m) ? ldg_u(static_cast<const UT*>(g.U) + (long long)t * g.ld + x) : 0.0f;
                    }
                    float v[32];  // [0, 16): r^2, [16, 32): u^2 of the block's 16 columns
#pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        const int t = col0 + blk * 16 + j;
                        const float rr = (xin && t < g.m) ? sum[blk * 16 + j] - u[j] : 0.0f;
                        v[j] = __fmul_rn(rr, rr);
                        v[16 + j] = __fmul_rn(u[j], u[j]);
                        pr += v[j];
                        pu += v[16 + j];
                    }
                    // column sums over the warp's 32 points: halving exchange, lane l ends with the sum of v[l]
#pragma unroll
                    for (int o = 16; o >= 1; o >>= 1) {
                        const bool hi = (lane & o) != 0;
#pragma unroll
                        for (int i = 0; i < o; ++i) {
                            const float send = hi ? v[i] : v[i + o];
                            const float keep = hi ? v[i + o] : v[i];
                            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, o);
                        }
                    }
                    prof[((q * 2 + c) * 4 + blk) * 32 + lane] = v[0];
                }
                float* pts = prof + 4 * 2 * 4 * 32;
                if (c == 1) { pts[row] = pr; pts[128 + row] = pu; }
                asm volatile("bar.sync 1, %0;" ::"n"(EPI_WARPS * 32) : "memory");  // the epilogue warps only
                if (c == 0) {  // this tile's per-point partial: column half 0 + column half 1
                    float* dst = g.out + (long long)tn * 2 * g.rows_r;
                    dst[pl] = pr + pts[row];
                    dst[g.rows_r + pl] = pu + pts[128 + row];
                }
                {   // per snapshot: the four lane quadrants in order, in fp64, into this CTA's partial
                    const int e = (warp - 2) * 32 + lane;
                    const int ch = e >> 7, blk = (e >> 5) & 3, l = e & 31;
                    double sq = 0.0;
#pragma unroll
                    for (int qq = 0; qq < 4; ++qq) sq += (double)prof[((qq * 2 + ch) * 4 + blk) * 32 + l];
                    const int t = tn * BN + ch * 64 + blk * 16 + (l & 15);
                    double* dst = g.loss_part + ((long long)blockIdx.x * 2 + (l >> 4)) * g.mp + t;
                    *dst += sq;
                }
            } else if (kPrune) {
                // GEMM 1 transposed: rows = snapshots, columns = points of the chunk.  r_0 = Rec - U exactly as EPI_RESID forms it; step
                // s = 1 .. steps peels term order[s - 1] off, r_s = r_{s-1} - a_s(x) b_s(t) (one FFMA), and sum_x r_s^2 over this
                // thread's 64 points is a running sum in registers: no cross-lane reduction, and a_s(x) is a broadcast read of the warp.
                const int t = tm * BM + row;
                const bool tin = t < g.m;
                const long long xc = g.x0 + (long long)tn * BN + c * 64;  // first point of this thread's columns
                float* a_s = reinterpret_cast<float*>(smem + NSTAGE * STAGE);
                float* p_s = a_s + kPruneSteps * BN;
                const int e = (warp - 2) * 32 + lane;  // 0 .. 255 over the epilogue warps
                const UT* up = static_cast<const UT*>(g.U) + (long long)t * g.ld + xc;
                float pu = 0.0f;
#pragma unroll
                for (int blk = 0; blk < 8; ++blk) {
                    float u[8];
                    ldg8_u(up + blk * 8, tin, u);
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const bool in = tin && xc + blk * 8 + j < g.n;
                        const float uu = in ? u[j] : 0.0f;
                        sum[blk * 8 + j] = in ? sum[blk * 8 + j] - uu : 0.0f;
                        pu = fmaf(uu, uu, pu);
                    }
                }
                const int nout = g.steps + 1;
                for (int o0 = 0; o0 < nout; o0 += kPruneSteps) {
                    const int nc = min(kPruneSteps, nout - o0);
                    float bv[kPruneSteps];
#pragma unroll
                    for (int i = 0; i < kPruneSteps; ++i) bv[i] = i < nc ? __ldg(g.prune_b + (long long)(o0 + i) * g.mp + t) : 0.0f;
                    // a of the chunk's steps at the tile's 128 points
#pragma unroll
                    for (int q4 = 0; q4 < kPruneSteps * BN / 4 / (EPI_WARPS * 32); ++q4) {
                        const int f = e + q4 * EPI_WARPS * 32, i = f / (BN / 4), x4 = f - i * (BN / 4);
                        float4 v = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
                        if (i < nc) v = __ldg(reinterpret_cast<const float4*>(g.prune_a + (long long)(o0 + i) * g.rows_r + (long long)tn * BN) + x4);
                        reinterpret_cast<float4*>(a_s)[f] = v;
                    }
                    asm volatile("bar.sync 1, %0;" ::"n"(EPI_WARPS * 32) : "memory");  // the epilogue warps only
#pragma unroll
                    for (int i = 0; i < kPruneSteps; ++i) {
                        if (i < nc) {
                            const uint32_t a = smem_u32(a_s + i * BN + c * 64);
                            float acc[8];
#pragma unroll
                            for (int j = 0; j < 8; ++j) acc[j] = 0.0f;
#pragma unroll
                            for (int j = 0; j < 64; j += 4) {
                                const float4 av = lds_v4(a + j * 4);  // the same address in every lane: a broadcast
                                sum[j] = fmaf(-av.x, bv[i], sum[j]);
                                sum[j + 1] = fmaf(-av.y, bv[i], sum[j + 1]);
                                sum[j + 2] = fmaf(-av.z, bv[i], sum[j + 2]);
                                sum[j + 3] = fmaf(-av.w, bv[i], sum[j + 3]);
#pragma unroll
                                for (int k = 0; k < 4; ++k) acc[(j + k) & 7] = fmaf(sum[j + k], sum[j + k], acc[(j + k) & 7]);
                            }
                            p_s[(c * (kPruneSteps + 1) + i) * BM + row] = ((acc[0] + acc[1]) + (acc[2] + acc[3])) + ((acc[4] + acc[5]) + (acc[6] + acc[7]));
                        }
                    }
                    if (o0 == 0) p_s[(c * (kPruneSteps + 1) + kPruneSteps) * BM + row] = pu;
                    asm volatile("bar.sync 1, %0;" ::"n"(EPI_WARPS * 32) : "memory");
                    // fp64: column half 0 + column half 1, added into this CTA's running partial [steps + 2][BM] (row steps + 1: sum_x u^2).
                    // Each element always falls to the same thread, so the partial needs no atomics.
                    const int nrow = nc + (o0 == 0 ? 1 : 0);
                    for (int f = e; f < nrow * BM; f += EPI_WARPS * 32) {
                        const int i = f / BM, tt = f - i * BM;
                        const int slot = i < nc ? i : kPruneSteps, o = i < nc ? o0 + i : nout;
                        double* dst = g.loss_part + ((long long)blockIdx.x * (nout + 1) + o) * BM + tt;
                        *dst += (double)p_s[slot * BM + tt] + (double)p_s[(kPruneSteps + 1 + slot) * BM + tt];
                    }
                }
            } else if (kGram) {
                // rows = snapshots t1 of tile tm, columns = snapshots t2 of tile tn >= tm: this slice's fp64 partial of the tile, accumulated
                // over the chunks in chunk order.  Stored [t2][t1] so that the 32 lanes of a warp write 32 consecutive doubles; every element
                // always falls to the same thread (the slice layout is the same for every chunk), so no atomics.
                double* Co = g.loss_part + ((long long)slice * g.tiles_n + rem) * (BM * BN) + row;
#pragma unroll
                for (int j = 0; j < 64; ++j) {
                    double* dst = Co + (long long)(c * 64 + j) * BM;
                    *dst = g.first_chunk ? (double)sum[j] : *dst + (double)sum[j];
                }
            } else {  // EPI_E: rows = snapshots, columns = library terms; this slice's partial of E^T, accumulated over the chunks
                const int t = tm * BM + row;
                float* Eo = g.Epart + (long long)slice * g.Kp * g.mld;
#pragma unroll
                for (int j = 0; j < 64; ++j) {
                    const int k = col0 + j;
                    if (k < g.Kp && t < g.mld) {
                        float* dst = Eo + (long long)k * g.mld + t;
                        const float v = (k < g.K && t < g.m) ? sum[j] : 0.0f;
                        *dst = g.first_chunk ? v : *dst + v;
                    }
                }
            }
        }
        if (kResid) {
            loss_acc = warp_sum(loss_acc);
            if (lane == 0) loss_s[warp - 2] = loss_acc;
        }
        tc_fence_before();
    }
    __syncthreads();
    if (kResid && tid == 0) {
        double s = 0.0;
        for (int i = 0; i < EPI_WARPS; ++i) s += loss_s[i];
        g.loss_part[blockIdx.x] = g.first_chunk ? s : g.loss_part[blockIdx.x] + s;
    }
    if (warp == 0) {
        tc_fence_after();
        tmem_dealloc<256>(tmem);
    }
}

// ------------------------------------------------------------------------------------------------- library terms for any (r, p)
// Column order of POOL_DATA (CYL:376-434) = combinations with replacement of range(r), degree by degree, lexicographic.  The index tuple of
// column j is found by unranking (no table upload, no host state: the kernel is stateless and capturable).
// Library columns may be a compact list: column c is term cols[c] of the K order (an active set, desmo_active_terms_prepare: strictly
// increasing, so the polynomial terms come first); cols == null is the whole library, column c = term c.  Entry j of the table then
// describes column j.
struct TermTable {
    uint8_t* idx;  // [T][8]: idx[j][0..deg) = mode indices multiplied left to right
    uint8_t* deg;  // [T]
};
__device__ __forceinline__ int term_of(const int32_t* __restrict__ cols, int c) { return cols ? cols[c] : c; }
__device__ __forceinline__ unsigned long long binom_d(int n, int k) {
    if (k < 0 || k > n) return 0ull;
    unsigned long long v = 1;
    for (int i = 1; i <= k; ++i) v = v * (unsigned long long)(n - k + i) / (unsigned long long)i;
    return v;
}
__global__ void term_table_kernel(int r, int p, int T, TermTable tab, const int32_t* __restrict__ cols, int ncols) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= T || j >= ncols) return;
    const int k = term_of(cols, j);
    if (k >= T) return;
    // degree of term k: first d with sum_{e<=d} C(r+e-1, e) > k
    long long rem = k;
    int d = 0;
    for (; d <= p; ++d) {
        const long long c = (long long)binom_d(r + d - 1, d);
        if (rem < c) break;
        rem -= c;
    }
    tab.deg[j] = (uint8_t)d;
    int prev = 0;
    for (int pos = 0; pos < d; ++pos) {
        // smallest v >= prev such that rem < #multisets of size d-pos-1 over values >= v ... summed from prev
        int v = prev;
        for (;; ++v) {
            const int left = d - pos - 1;
            const long long c = (long long)binom_d((r - v) + left - 1, left);  // multisets of size `left` from the r - v values >= v
            if (rem < c) break;
            rem -= c;
        }
        tab.idx[j * 8 + pos] = (uint8_t)v;
        prev = v;
    }
    for (int pos = d; pos < 8; ++pos) tab.idx[j * 8 + pos] = 0;
}

// G planes of a chunk: thread <-> point, loop over the K columns.  Gp[plane][k][xl], xl contiguous; rows K..Kr-1 and columns of points >= n are zero.
// (K here counts the columns: the library's K, or the active set's size with cols its list)
__global__ void __launch_bounds__(256) library_planes_kernel(const float* __restrict__ P, const float* __restrict__ phi,
                                                             const float* __restrict__ omega, TermTable tab, const int32_t* __restrict__ cols,
                                                             int r, int T, int K, int Kr, long long n, long long ld, long long x0,
                                                             long long rows_c, __nv_bfloat16* __restrict__ Gp) {
    const long long xl = (long long)blockIdx.x * 256 + threadIdx.x;
    if (xl >= rows_c) return;
    const long long x = x0 + xl;
    const bool xin = x < n;
    float lat[DESMO_MAX_R];
    for (int i = 0; i < r; ++i) lat[i] = xin ? phi[(long long)i * ld + x] * P[(long long)i * ld + x] : 0.0f;
    const size_t plane = (size_t)Kr * rows_c;
    for (int k = blockIdx.y; k < Kr; k += gridDim.y) {
        float v = 0.0f;
        const int term = k < K ? term_of(cols, k) : K;
        if (xin) {
            if (term < T) {
                const int deg = tab.deg[k];
                v = 1.0f;
                for (int q = 0; q < deg; ++q) {
                    const float f = lat[tab.idx[k * 8 + q]];
                    v = (q == 0) ? f : v * f;  // left-to-right products, as CYL:390-431
                }
            } else if (k < K) {
                const int b = (term - T) / r, i = (term - T) - b * r;
                const float arg = omega[3 * i + b] * lat[i];
                v = (b == 0) ? sinf(arg) : (b == 1) ? cosf(arg) : tanhf(arg);
            }
        }
        const __nv_bfloat16 b1 = __float2bfloat16_rn(v);
        const float e1 = v - __bfloat162float(b1);
        const __nv_bfloat16 b2 = __float2bfloat16_rn(e1);
        const __nv_bfloat16 b3 = __float2bfloat16_rn(e1 - __bfloat162float(b2));
        const size_t o = (size_t)k * rows_c + xl;
        Gp[o] = b1;
        Gp[plane + o] = b2;
        Gp[2 * plane + o] = b3;
    }
}

// W planes [3][Kr][mp] from the fp32 W [Kp][mld] of desmo_build_w (rows >= K and columns >= m are zero); row k is W's row cols[k]
__global__ void __launch_bounds__(256) w_planes_kernel(const float* __restrict__ W, const int32_t* __restrict__ cols, int K, int Kr, int m,
                                                       int mld, int mp, __nv_bfloat16* __restrict__ Wp) {
    const int k = blockIdx.x;
    const size_t plane = (size_t)Kr * mp;
    const size_t src = k < K ? (size_t)term_of(cols, k) * mld : 0;
    for (int t = threadIdx.x; t < mp; t += 256) {
        const float w = (k < K && t < m) ? W[src + t] : 0.0f;
        const __nv_bfloat16 b1 = __float2bfloat16_rn(w);
        const float e1 = w - __bfloat162float(b1);
        const __nv_bfloat16 b2 = __float2bfloat16_rn(e1);
        const __nv_bfloat16 b3 = __float2bfloat16_rn(e1 - __bfloat162float(b2));
        const size_t o = (size_t)k * mp + t;
        Wp[o] = b1;
        Wp[plane + o] = b2;
        Wp[2 * plane + o] = b3;
    }
}

// Chain rule D -> d mse / d phi, d mse / d omega for any (r, p): thread <-> point, one pass over the library columns.  For column
// j = Phi_{i1} ... Phi_{id}: d L_j / d Phi_v = sum over the positions holding v of the product of the other factors (multiplicity-aware,
// the same formula as the oracle's pool_data_derivative).  dom_part[cta][3r] are per-CTA partial sums of d omega.  Dacc row c is library
// column c: term cols[c] of an active set of Ka terms, pos[k] = the column of term k or -1 (both null: the whole library, Ka = K).
__global__ void __launch_bounds__(128) chain_rule_generic_kernel(const float* __restrict__ Dacc, const float* __restrict__ P,
                                                                 const float* __restrict__ phi, const float* __restrict__ omega, TermTable tab,
                                                                 const int32_t* __restrict__ cols, const int32_t* __restrict__ pos, int Ka,
                                                                 int r, int T, long long n, long long ld, float scale, float* __restrict__ dphi,
                                                                 double* __restrict__ dom_part) {
    extern __shared__ double dom_s[];  // [3r]
    const int tid = threadIdx.x, lane = tid & 31;
    for (int i = tid; i < 3 * r; i += 128) dom_s[i] = 0.0;
    __syncthreads();
    const long long ntiles = (ld + 127) / 128;
    for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const long long x = tile * 128 + tid;
        const bool xin = x < n;
        float lat[DESMO_MAX_R], dl[DESMO_MAX_R];
        for (int i = 0; i < r; ++i) {
            lat[i] = (x < ld) ? phi[(long long)i * ld + x] * P[(long long)i * ld + x] : 0.0f;
            dl[i] = 0.0f;
        }
        if (xin) {
            for (int j = 0; j < Ka && term_of(cols, j) < T; ++j) {  // the active polynomial columns; the constant has no derivative
                const int deg = tab.deg[j];
                if (deg == 0) continue;
                const float dj = Dacc[(long long)j * ld + x];
                for (int pos = 0; pos < deg; ++pos) {
                    float rest = 1.0f;
                    for (int q = 0; q < deg; ++q)
                        if (q != pos) rest *= lat[tab.idx[j * 8 + q]];
                    dl[tab.idx[j * 8 + pos]] += dj * rest;
                }
            }
        }
        for (int i = 0; i < r; ++i) {
            const float ph = lat[i];
            const float ws = omega[3 * i], wc = omega[3 * i + 1], wh = omega[3 * i + 2];
            float ds = 0.0f, dc = 0.0f, dh = 0.0f;
            if (xin) {  // an absent trig term has no column: its dL/dG is zero
                const int cs_ = pos ? pos[T + i] : T + i, cc_ = pos ? pos[T + r + i] : T + r + i, ch_ = pos ? pos[T + 2 * r + i] : T + 2 * r + i;
                if (cs_ >= 0) ds = Dacc[(long long)cs_ * ld + x];
                if (cc_ >= 0) dc = Dacc[(long long)cc_ * ld + x];
                if (ch_ >= 0) dh = Dacc[(long long)ch_ * ld + x];
            }
            const float cs = cosf(ws * ph), sn = sinf(wc * ph), th = tanhf(wh * ph);
            const float sech2 = 1.0f - th * th;
            const float g = dl[i] + (ds * ws * cs - dc * wc * sn + dh * wh * sech2);
            if (x < ld) dphi[(long long)i * ld + x] = xin ? scale * g * P[(long long)i * ld + x] : 0.0f;
            const float o0 = warp_sum(ds * ph * cs), o1 = warp_sum(-dc * ph * sn), o2 = warp_sum(dh * ph * sech2);
            if (lane == 0) {
                atomicAdd(&dom_s[3 * i], (double)o0);
                atomicAdd(&dom_s[3 * i + 1], (double)o1);
                atomicAdd(&dom_s[3 * i + 2], (double)o2);
            }
        }
    }
    __syncthreads();
    for (int i = tid; i < 3 * r; i += 128) dom_part[(long long)blockIdx.x * 3 * r + i] = dom_s[i] * (double)scale;
}

// Phi^T Phi (r x r) partial sums: CTA tile of 128 points in shared memory, thread <-> pairs (i <= j).
__global__ void __launch_bounds__(256) gram_phi_kernel(const float* __restrict__ P, const float* __restrict__ phi, int r, long long n,
                                                       long long ld, double* __restrict__ gram_part) {
    extern __shared__ float lat_s[];  // [r][129]
    const int tid = threadIdx.x;
    const int npairs = r * (r + 1) / 2;
    constexpr int kMaxPer = (DESMO_MAX_R * (DESMO_MAX_R + 1) / 2 + 255) / 256;
    float acc[kMaxPer];
#pragma unroll
    for (int i = 0; i < kMaxPer; ++i) acc[i] = 0.0f;
    const long long ntiles = (n + 127) / 128;
    for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        __syncthreads();
        for (int e = tid; e < r * 128; e += 256) {
            const int i = e >> 7, xx = e & 127;
            const long long x = tile * 128 + xx;
            lat_s[i * 129 + xx] = (x < n) ? phi[(long long)i * ld + x] * P[(long long)i * ld + x] : 0.0f;
        }
        __syncthreads();
#pragma unroll
        for (int s = 0; s < kMaxPer; ++s) {
            const int pr = tid + s * 256;
            if (pr < npairs) {
                // pair index -> (i, j), i <= j, row-major over the upper triangle
                int i = 0, rem = pr;
                while (rem >= r - i) { rem -= r - i; ++i; }
                const int j = i + rem;
                float a = 0.0f;
                for (int xx = 0; xx < 128; ++xx) a = fmaf(lat_s[i * 129 + xx], lat_s[j * 129 + xx], a);
                acc[s] += a;
            }
        }
    }
#pragma unroll
    for (int s = 0; s < kMaxPer; ++s) {
        const int pr = tid + s * 256;
        if (pr < npairs) gram_part[(long long)blockIdx.x * npairs + pr] = (double)acc[s];
    }
}

// Fixed-order sums of all partials into `red` = [E (Kp x mld) | sum r^2 | Phi^T Phi (r x r) | d omega (3r)].  The slices of Epart hold
// the library columns ([nslice][ecount_c / mld][mld]); row k of E is column pos[k] (pos null: column k), zero for an absent term.
__global__ void __launch_bounds__(256) reduce_generic_kernel(const float* __restrict__ Epart, int nslice, long long ecount, long long ecount_c,
                                                             const int32_t* __restrict__ pos, int K, int mld,
                                                             const double* __restrict__ loss_part, int nloss, const double* __restrict__ gram_part,
                                                             int ngram, const double* __restrict__ dom_part, int ndom, int r,
                                                             float* __restrict__ red) {
    const long long o = (long long)blockIdx.x * 256 + threadIdx.x;
    if (o < ecount) {
        const int k = (int)(o / mld), t = (int)(o - (long long)k * mld);
        const int c = k < K ? (pos ? pos[k] : k) : -1;
        float s = 0.0f;
        if (c >= 0)
            for (int b = 0; b < nslice; ++b) s += Epart[(long long)b * ecount_c + (long long)c * mld + t];
        red[o] = s;
    }
    if (blockIdx.x == 0) {
        const int npairs = r * (r + 1) / 2;
        if (threadIdx.x == 0) {
            double s = 0.0;
            for (int b = 0; b < nloss; ++b) s += loss_part[b];
            red[ecount] = (float)s;
        }
        for (int pr = threadIdx.x; pr < npairs; pr += 256) {
            double s = 0.0;
            for (int b = 0; b < ngram; ++b) s += gram_part[(long long)b * npairs + pr];
            int i = 0, rem = pr;
            while (rem >= r - i) { rem -= r - i; ++i; }
            const int j = i + rem;
            red[ecount + 1 + i * r + j] = (float)s;
            red[ecount + 1 + j * r + i] = (float)s;
        }
        for (int w = threadIdx.x; w < 3 * r; w += 256) {
            double s = 0.0;
            for (int b = 0; b < ndom; ++b) s += dom_part[(long long)b * 3 * r + w];
            red[ecount + 1 + r * r + w] = (float)s;
        }
    }
}

// Squared column norms of the library for any K (post-hoc norms): thread <-> point, warp reduction + one atomic per warp and column.
__global__ void __launch_bounds__(256) colnorm2_generic_kernel(const float* __restrict__ P, const float* __restrict__ phi,
                                                               const float* __restrict__ omega, TermTable tab, int r, int T, int K, long long n,
                                                               long long ld, float* __restrict__ out) {
    const long long x = (long long)blockIdx.x * 256 + threadIdx.x;
    const bool xin = x < n;
    float lat[DESMO_MAX_R];
    for (int i = 0; i < r; ++i) lat[i] = xin ? (P ? phi[(long long)i * ld + x] * P[(long long)i * ld + x] : phi[(long long)i * ld + x]) : 0.0f;
    for (int k = 0; k < K; ++k) {
        float v = 0.0f;
        if (xin) {
            if (k < T) {
                const int deg = tab.deg[k];
                v = 1.0f;
                for (int q = 0; q < deg; ++q) {
                    const float f = lat[tab.idx[k * 8 + q]];
                    v = (q == 0) ? f : v * f;
                }
            } else {
                const int b = (k - T) / r, i = (k - T) - b * r;
                const float arg = omega[3 * i + b] * lat[i];
                v = (b == 0) ? sinf(arg) : (b == 1) ? cosf(arg) : tanhf(arg);
            }
        }
        const float s = warp_sum(v * v);
        if ((threadIdx.x & 31) == 0 && s != 0.0f) atomicAdd(out + k, s);
    }
}

// ------------------------------------------------------------------------------------------------- host side
// 2-D bf16 map over `rows` rows of `inner` contiguous elements; box = [64 inner][box_rows]
static int make_map(CUtensorMap* tm, const void* base, long long inner, long long rows, int box_rows) {
    EncodeTiledFn enc = encode_fn();
    if (!enc) { set_error("cuTensorMapEncodeTiled not available"); return DESMO_ERR_CUDA; }
    const cuuint64_t dims[2] = {(cuuint64_t)inner, (cuuint64_t)rows};
    const cuuint64_t strides[1] = {(cuuint64_t)inner * 2};
    const cuuint32_t box[2] = {64, (cuuint32_t)box_rows};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult cr = enc(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (cr != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed (%d) inner=%lld rows=%lld", (int)cr, inner, rows); return DESMO_ERR_CUDA; }
    return DESMO_OK;
}

template <bool A_MN, bool B_MN, int NPA, int NPB, int EPI>
static int launch_gemm(const GemmArgs& g, const CUtensorMap& tmA, const CUtensorMap& tmB, int sms, cudaStream_t st) {
    constexpr size_t stage = (size_t)(NPA + NPB) * PLANE_TILE;
    constexpr int nstage = (NPA + NPB) >= 6 ? 2 : 3;
    constexpr size_t extra = (EPI == EPI_PROFILE || EPI == EPI_PROFILE_BF16) ? kProfSmem : (EPI == EPI_PRUNE || EPI == EPI_PRUNE_BF16) ? kPruneSmem : 0;
    const size_t smem = nstage * stage + 1024 + extra;
    auto kern = gemm_planes_kernel<A_MN, B_MN, NPA, NPB, EPI>;
    DESMO_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int items = g.tiles_m * g.tiles_n * g.nslice;
    const int grid = items < sms ? items : sms;
    kern<<<grid, THREADS, smem, st>>>(g, tmA, tmB);
    DESMO_CUDA(cudaGetLastError());
    return DESMO_OK;
}

}  // namespace gp

static size_t align_up_g(size_t v, size_t a) { return (v + a - 1) / a * a; }

// Workspace of the general path, carved from the caller's buffer behind the fused kernels' regions.
struct GemmWorkspace {
    uint8_t* tab_idx; uint8_t* tab_deg;
    __nv_bfloat16* Gp;   // [3][Kr][rows_c]
    __nv_bfloat16* Wp;   // [3][Kr][mp]
    __nv_bfloat16* Rp;   // [2][rows_c][mp]
    float* Epart;        // [nslice_max][Kp][mld]
    double* loss_part;   // [sms]
    double* gram_part;   // [kGramCtas][r(r+1)/2]
    double* dom_part;    // [kChainCtas][3r]
    size_t bytes;
};
constexpr int kGramCtas = 148, kChainCtas = 296, kSliceMax = 32;

static void gemm_dims(const desmo_shape* s, int K, int* Kr, int* mp, long long* rows_c) {
    *Kr = (K + 127) / 128 * 128;
    *mp = (s->m + 127) / 128 * 128;
    long long rc = s->ld < gp::kChunkPoints ? s->ld : gp::kChunkPoints;
    *rows_c = (rc + 127) / 128 * 128;
}

size_t gemm_workspace_bytes(const desmo_shape* s, int T, int K, int Kp, uint8_t* base, GemmWorkspace* w) {
    int Kr, mp;
    long long rows_c;
    gemm_dims(s, K, &Kr, &mp, &rows_c);
    size_t off = 0;
    auto take = [&](size_t bytes) { uint8_t* p = base ? base + off : nullptr; off = align_up_g(off + bytes, 1024); return p; };
    GemmWorkspace g{};
    g.tab_idx = take((size_t)T * 8);
    g.tab_deg = take((size_t)T);
    g.Gp = reinterpret_cast<__nv_bfloat16*>(take((size_t)3 * Kr * rows_c * 2));
    g.Wp = reinterpret_cast<__nv_bfloat16*>(take((size_t)3 * Kr * mp * 2));
    g.Rp = reinterpret_cast<__nv_bfloat16*>(take((size_t)2 * rows_c * mp * 2));
    g.Epart = reinterpret_cast<float*>(take((size_t)kSliceMax * Kp * s->mld * 4));
    g.loss_part = reinterpret_cast<double*>(take(sizeof(double) * 1024));
    g.gram_part = reinterpret_cast<double*>(take(sizeof(double) * kGramCtas * (size_t)(s->r * (s->r + 1) / 2)));
    g.dom_part = reinterpret_cast<double*>(take(sizeof(double) * kChainCtas * 3 * (size_t)s->r));
    g.bytes = off;
    if (w) *w = g;
    return off;
}

// supplied = true: U holds dL/drecon and R := (n_global m / 2) U -- not fused here: the general path forms R planes from U by an
// elementwise kernel instead of GEMM 1.
__global__ void __launch_bounds__(256) supplied_planes_kernel(const float* __restrict__ U, long long n, long long ld, long long x0,
                                                              long long rows_c, int m, int mp, float seed, __nv_bfloat16* __restrict__ Rp) {
    // thread <-> (point, 8 snapshots): reads are strided by ld (evaluation path; not bandwidth-critical)
    const long long xl = (long long)blockIdx.x * 256 + threadIdx.x;
    if (xl >= rows_c) return;
    const long long x = x0 + xl;
    for (int t0 = blockIdx.y * 8; t0 < mp; t0 += gridDim.y * 8) {
        uint32_t w1[4], w2[4];
#pragma unroll
        for (int j = 0; j < 8; j += 2) {
            const int t = t0 + j;
            const float r0 = (x < n && t < m) ? seed * U[(long long)t * ld + x] : 0.0f;
            const float r1 = (x < n && t + 1 < m) ? seed * U[(long long)(t + 1) * ld + x] : 0.0f;
            gp::split2_pair(r0, r1, w1[j >> 1], w2[j >> 1]);
        }
        uint4* d0 = reinterpret_cast<uint4*>(Rp + xl * mp + t0);
        uint4* d1 = reinterpret_cast<uint4*>(Rp + (rows_c + xl) * mp + t0);
        *d0 = make_uint4(w1[0], w1[1], w1[2], w1[3]);
        *d1 = make_uint4(w2[0], w2[1], w2[2], w2[3]);
    }
}

int fused_gemm_path(const desmo_shape* s, int T, int K, int Kp, const void* U, int u_dtype, const float* P, const float* phi, const float* omega,
                    const float* W, float* dphi, float* red, float* Dacc, void* gemm_ws, cudaStream_t st, bool supplied,
                    const int32_t* active, int Ka) {
    using namespace gp;
    int dev = 0, sms = 0;
    DESMO_CUDA(cudaGetDevice(&dev));
    DESMO_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    GemmWorkspace w;
    gemm_workspace_bytes(s, T, K, Kp, static_cast<uint8_t*>(gemm_ws), &w);
    // Library columns: the active set (pos [K] = column of each term or -1, then cols [Ka] = the terms) or, without one, all K terms.
    // The workspace is laid out for K; the planes, GEMM extents and partials below use the Ka columns only.
    const int32_t* pos = active;
    const int32_t* cols = active ? active + K : nullptr;
    if (!active) Ka = K;
    const int Kap = (Ka + 15) / 16 * 16;
    int Kr, mp;
    long long rows_c;
    gemm_dims(s, Ka, &Kr, &mp, &rows_c);
    const int r = s->r;
    TermTable tab{w.tab_idx, w.tab_deg};
    term_table_kernel<<<(T + 127) / 128, 128, 0, st>>>(r, s->polyorder, T, tab, cols, Ka);
    w_planes_kernel<<<Kr, 256, 0, st>>>(W, cols, Ka, Kr, s->m, s->mld, mp, w.Wp);
    DESMO_CUDA(cudaGetLastError());

    CUtensorMap tmG_mn, tmG_k, tmW_mn, tmW_k, tmR_k, tmR_mn;
    int rc;
    // G planes [3*Kr rows][rows_c]: MN-major A of GEMM 1 (box 64 x 64), K-major B of GEMM 4 (box 64 x 128)
    if ((rc = make_map(&tmG_mn, w.Gp, rows_c, 3LL * Kr, 64))) return rc;
    if ((rc = make_map(&tmG_k, w.Gp, rows_c, 3LL * Kr, 128))) return rc;
    // W planes [3*Kr rows][mp]: MN-major B of GEMM 1, K-major B of GEMM 3
    if ((rc = make_map(&tmW_mn, w.Wp, mp, 3LL * Kr, 64))) return rc;
    if ((rc = make_map(&tmW_k, w.Wp, mp, 3LL * Kr, 128))) return rc;
    // R planes [2*rows_c rows][mp]: K-major A of GEMM 3, MN-major A of GEMM 4
    if ((rc = make_map(&tmR_k, w.Rp, mp, 2LL * rows_c, 128))) return rc;
    if ((rc = make_map(&tmR_mn, w.Rp, mp, 2LL * rows_c, 64))) return rc;

    const int n_lib16 = Kap;
    const float seed = (float)(0.5 * (double)s->n_global * (double)s->m);
    int nslice_used = 1, nloss = 0;
    bool first = true;
    for (long long x0 = 0; x0 < s->ld; x0 += rows_c, first = false) {
        const long long pts = (s->ld - x0 < rows_c) ? s->ld - x0 : rows_c;  // multiple of 128 (ld is a multiple of 256)
        const int tiles_p = (int)(pts / 128);
        {
            dim3 grid((unsigned)((rows_c + 255) / 256), (unsigned)(Kr < 64 ? Kr : 64));
            library_planes_kernel<<<grid, 256, 0, st>>>(P, phi, omega, tab, cols, r, T, Ka, Kr, s->n, s->ld, x0, rows_c, w.Gp);
            DESMO_CUDA(cudaGetLastError());
        }
        GemmArgs g{};
        g.U = U; g.Rp = w.Rp; g.Dacc = Dacc; g.Epart = w.Epart; g.loss_part = w.loss_part;
        g.n = s->n; g.ld = s->ld; g.x0 = x0; g.rows_r = rows_c; g.m = s->m; g.mld = s->mld; g.mp = mp; g.K = Ka; g.Kp = Kap;
        g.first_chunk = first ? 1 : 0; g.n_lib16 = n_lib16;
        if (!supplied) {
            // GEMM 1: Rec[p x t] = G W; A = G (MN-major: p contiguous), B = W (MN-major: t contiguous), contraction over the library
            g.tiles_m = tiles_p; g.tiles_n = mp / 128; g.nslice = 1; g.kblocks = (Ka + 63) / 64; g.kb_per_slice = g.kblocks; g.kgroup = 4;
            g.a_rows = Kr; g.b_rows = Kr;
            rc = u_dtype == DESMO_DTYPE_BF16 ? launch_gemm<true, true, 3, 3, EPI_RESID_BF16>(g, tmG_mn, tmW_mn, sms, st)
                                             : launch_gemm<true, true, 3, 3, EPI_RESID>(g, tmG_mn, tmW_mn, sms, st);
            if (rc) return rc;
            const int items = g.tiles_m * g.tiles_n;
            nloss = nloss > (items < sms ? items : sms) ? nloss : (items < sms ? items : sms);
        } else {
            dim3 grid((unsigned)((rows_c + 255) / 256), 16);
            if (u_dtype != DESMO_DTYPE_F32) { set_error("GEMM path: recon_backward takes an fp32 upstream gradient"); return DESMO_ERR_ARG; }
            supplied_planes_kernel<<<grid, 256, 0, st>>>(static_cast<const float*>(U), s->n, s->ld, x0, rows_c, s->m, mp, seed, w.Rp);
            DESMO_CUDA(cudaGetLastError());
        }
        // GEMM 3: D[p x lib] = R W^T; A = R (K-major: t contiguous), B = W (K-major), contraction over the snapshots
        g.tiles_m = tiles_p; g.tiles_n = (Ka + 127) / 128; g.nslice = 1; g.kblocks = mp / 64; g.kb_per_slice = g.kblocks; g.kgroup = 32;
        g.a_rows = (int)rows_c; g.b_rows = Kr;
        if ((rc = launch_gemm<false, false, 2, 2, EPI_D>(g, tmR_k, tmW_k, sms, st))) return rc;
        // GEMM 4: E^T[t x lib] = R^T G; A = R (MN-major: t contiguous), B = G (K-major: p contiguous), contraction over the chunk's points
        g.tiles_m = mp / 128; g.tiles_n = (Ka + 127) / 128; g.kblocks = (int)(pts / 64);
        {
            const int tiles = g.tiles_m * g.tiles_n;
            int ns = sms / tiles;
            if (ns < 1) ns = 1;
            if (ns > kSliceMax) ns = kSliceMax;
            if (ns > g.kblocks) ns = g.kblocks;
            // all chunks must use the same slice layout (partials accumulate slot by slot): fix it by the first (largest) chunk
            if (first) nslice_used = ns;
            g.nslice = nslice_used;
            g.kb_per_slice = (g.kblocks + g.nslice - 1) / g.nslice;
            if (g.kb_per_slice < 1) g.kb_per_slice = 1;
        }
        g.kgroup = 32;
        g.a_rows = (int)rows_c; g.b_rows = Kr;
        if ((rc = launch_gemm<true, false, 2, 2, EPI_E>(g, tmR_mn, tmG_k, sms, st))) return rc;
    }
    // chain rule, Phi^T Phi, final sums
    const float scale = (float)(2.0 / ((double)s->n_global * (double)s->m));
    const long long ntiles = (s->ld + 127) / 128;
    const int gc = (int)(ntiles < kChainCtas ? ntiles : kChainCtas);
    chain_rule_generic_kernel<<<gc, 128, sizeof(double) * 3 * r, st>>>(Dacc, P, phi, omega, tab, cols, pos, Ka, r, T, s->n, s->ld, scale, dphi,
                                                                        w.dom_part);
    const long long gtiles = (s->n + 127) / 128;
    const int gg = (int)(gtiles < kGramCtas ? gtiles : kGramCtas);
    const size_t gsm = sizeof(float) * (size_t)r * 129;
    DESMO_CUDA(cudaFuncSetAttribute(gram_phi_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gsm));
    gram_phi_kernel<<<gg, 256, gsm, st>>>(P, phi, r, s->n, s->ld, w.gram_part);
    const long long ecount = (long long)Kp * s->mld;
    reduce_generic_kernel<<<(unsigned)((ecount + 255) / 256), 256, 0, st>>>(w.Epart, nslice_used, ecount, (long long)Kap * s->mld, pos, K, s->mld,
                                                                            w.loss_part, supplied ? 0 : nloss, w.gram_part, gg, w.dom_part, gc, r,
                                                                            red);
    DESMO_CUDA(cudaGetLastError());
    return DESMO_OK;
}

// Materialised reconstruction for any K: library planes + GEMM 1 with the plain store epilogue (evaluation only; scratch comes from
// the stream-ordered allocator because desmo_reconstruct takes no workspace).
int reconstruct_gemm_path(const desmo_shape* s, int T, int K, int Kp, const float* P, const float* phi, const float* omega, const float* W,
                          float* out, cudaStream_t st) {
    using namespace gp;
    int dev = 0, sms = 0;
    DESMO_CUDA(cudaGetDevice(&dev));
    DESMO_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const size_t bytes = gemm_workspace_bytes(s, T, K, Kp, nullptr, nullptr);
    void* scratch = nullptr;
    DESMO_CUDA(cudaMallocAsync(&scratch, bytes, st));
    GemmWorkspace w;
    gemm_workspace_bytes(s, T, K, Kp, static_cast<uint8_t*>(scratch), &w);
    int Kr, mp;
    long long rows_c;
    gemm_dims(s, K, &Kr, &mp, &rows_c);
    TermTable tab{w.tab_idx, w.tab_deg};
    term_table_kernel<<<(T + 127) / 128, 128, 0, st>>>(s->r, s->polyorder, T, tab, nullptr, K);
    w_planes_kernel<<<Kr, 256, 0, st>>>(W, nullptr, K, Kr, s->m, s->mld, mp, w.Wp);
    CUtensorMap tmG_mn, tmW_mn;
    int rc;
    if ((rc = make_map(&tmG_mn, w.Gp, rows_c, 3LL * Kr, 64)) || (rc = make_map(&tmW_mn, w.Wp, mp, 3LL * Kr, 64))) { cudaFreeAsync(scratch, st); return rc; }
    for (long long x0 = 0; x0 < s->ld && !rc; x0 += rows_c) {
        const long long pts = (s->ld - x0 < rows_c) ? s->ld - x0 : rows_c;
        dim3 grid((unsigned)((rows_c + 255) / 256), (unsigned)(Kr < 64 ? Kr : 64));
        library_planes_kernel<<<grid, 256, 0, st>>>(P, phi, omega, tab, nullptr, s->r, T, K, Kr, s->n, s->ld, x0, rows_c, w.Gp);
        GemmArgs g{};
        g.out = out; g.n = s->n; g.ld = s->ld; g.x0 = x0; g.rows_r = rows_c; g.m = s->m; g.mld = s->mld; g.mp = mp; g.K = K; g.Kp = Kp;
        g.tiles_m = (int)(pts / 128); g.tiles_n = mp / 128; g.nslice = 1; g.kblocks = (K + 63) / 64; g.kb_per_slice = g.kblocks; g.kgroup = 4;
        g.a_rows = Kr; g.b_rows = Kr; g.first_chunk = 1;
        rc = launch_gemm<true, true, 3, 3, EPI_RECON>(g, tmG_mn, tmW_mn, sms, st);
    }
    cudaFreeAsync(scratch, st);
    return rc;
}

// Residual profile (desmo_residual_profile): library planes + GEMM 1 with the profile epilogue, then fixed-order sums of the partials.
// Points per chunk: the chunk's G planes and per-point partials take about kProfileChunkBytes, so that they stay in L2 while U streams.
constexpr size_t kProfileChunkBytes = 32u << 20;

// point[0][x] = sum_t r^2, point[1][x] = sum_t u^2 for the chunk's points: the tiles_n partials in order, in fp64, rounded once
__global__ void __launch_bounds__(256) profile_points_kernel(const float* __restrict__ pp, int tiles_n, long long rows_c, long long pts,
                                                             long long n, long long ld, long long x0, float* __restrict__ point) {
    const long long xl = (long long)blockIdx.x * 256 + threadIdx.x;
    if (xl >= pts) return;
    double a = 0.0, b = 0.0;
    for (int tn = 0; tn < tiles_n; ++tn) {
        a += (double)pp[(long long)(2 * tn) * rows_c + xl];
        b += (double)pp[(long long)(2 * tn + 1) * rows_c + xl];
    }
    const long long x = x0 + xl;
    point[x] = x < n ? (float)a : 0.0f;
    point[ld + x] = x < n ? (float)b : 0.0f;
}

// snap[q][t] = sum over the CTAs, in order, of their partials [nparts][2][mp]
__global__ void __launch_bounds__(256) profile_snapshots_kernel(const double* __restrict__ part, int nparts, int m, int mp,
                                                                double* __restrict__ snap) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= 2 * m) return;
    const int q = i / m, t = i - q * m;
    double s = 0.0;
    for (int b = 0; b < nparts; ++b) s += part[((long long)b * 2 + q) * mp + t];
    snap[i] = s;
}

int residual_profile_gemm_path(const desmo_shape* s, int T, int K, int Kp, const void* U, int u_dtype, const float* P, const float* phi,
                               const float* omega, const float* W, double* snap, float* point, cudaStream_t st) {
    using namespace gp;
    int dev = 0, sms = 0;
    DESMO_CUDA(cudaGetDevice(&dev));
    DESMO_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    // GEMM 1 reads (K + 63) / 64 k-blocks: planes of that many rows give the same products as reconstruct_gemm_path's
    const int Kr = (K + 63) / 64 * 64;
    const int mp = (s->m + 127) / 128 * 128, tiles_n = mp / 128;
    const size_t per_point = (size_t)3 * Kr * 2 + (size_t)tiles_n * 2 * 4;
    long long rows_c = (long long)(kProfileChunkBytes / per_point) / 128 * 128;
    if (rows_c < 128) rows_c = 128;
    if (rows_c > s->ld) rows_c = s->ld;
    size_t off = 0;
    auto take = [&](size_t bytes) { const size_t o = off; off = align_up_g(off + bytes, 1024); return o; };
    const size_t o_idx = take((size_t)T * 8), o_deg = take((size_t)T), o_gp = take((size_t)3 * Kr * rows_c * 2),
                 o_wp = take((size_t)3 * Kr * mp * 2), o_pp = take((size_t)tiles_n * 2 * rows_c * 4),
                 o_part = take((size_t)sms * 2 * mp * sizeof(double));
    uint8_t* scratch = nullptr;
    DESMO_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&scratch), off, st));
    __nv_bfloat16* Gp = reinterpret_cast<__nv_bfloat16*>(scratch + o_gp);
    __nv_bfloat16* Wp = reinterpret_cast<__nv_bfloat16*>(scratch + o_wp);
    float* pp = reinterpret_cast<float*>(scratch + o_pp);
    double* part = reinterpret_cast<double*>(scratch + o_part);
    TermTable tab{scratch + o_idx, scratch + o_deg};
    int rc = check_cuda(cudaMemsetAsync(part, 0, (size_t)sms * 2 * mp * sizeof(double), st), "cudaMemsetAsync");
    CUtensorMap tmG_mn, tmW_mn;
    if (!rc) {
        term_table_kernel<<<(T + 127) / 128, 128, 0, st>>>(s->r, s->polyorder, T, tab, nullptr, K);
        w_planes_kernel<<<Kr, 256, 0, st>>>(W, nullptr, K, Kr, s->m, s->mld, mp, Wp);
        rc = check_cuda(cudaGetLastError(), "w_planes_kernel");
    }
    if (!rc && !(rc = make_map(&tmG_mn, Gp, rows_c, 3LL * Kr, 64))) rc = make_map(&tmW_mn, Wp, mp, 3LL * Kr, 64);
    for (long long x0 = 0; x0 < s->ld && !rc; x0 += rows_c) {
        const long long pts = (s->ld - x0 < rows_c) ? s->ld - x0 : rows_c;  // multiple of 128
        dim3 grid((unsigned)((rows_c + 255) / 256), 64u);
        library_planes_kernel<<<grid, 256, 0, st>>>(P, phi, omega, tab, nullptr, s->r, T, K, Kr, s->n, s->ld, x0, rows_c, Gp);
        GemmArgs g{};
        g.U = U; g.out = pp; g.loss_part = part;
        g.n = s->n; g.ld = s->ld; g.x0 = x0; g.rows_r = rows_c; g.m = s->m; g.mld = s->mld; g.mp = mp; g.K = K; g.Kp = Kp;
        g.tiles_m = (int)(pts / 128); g.tiles_n = tiles_n; g.nslice = 1; g.kblocks = (K + 63) / 64; g.kb_per_slice = g.kblocks; g.kgroup = 4;
        g.a_rows = Kr; g.b_rows = Kr; g.first_chunk = 1;
        rc = u_dtype == DESMO_DTYPE_BF16 ? launch_gemm<true, true, 3, 3, EPI_PROFILE_BF16>(g, tmG_mn, tmW_mn, sms, st)
                                         : launch_gemm<true, true, 3, 3, EPI_PROFILE>(g, tmG_mn, tmW_mn, sms, st);
        if (rc) break;
        profile_points_kernel<<<(unsigned)((pts + 255) / 256), 256, 0, st>>>(pp, tiles_n, rows_c, pts, s->n, s->ld, x0, point);
        rc = check_cuda(cudaGetLastError(), "profile_points_kernel");
    }
    if (!rc) {
        profile_snapshots_kernel<<<(2 * s->m + 255) / 256, 256, 0, st>>>(part, sms, s->m, mp, snap);
        rc = check_cuda(cudaGetLastError(), "profile_snapshots_kernel");
    }
    cudaFreeAsync(scratch, st);
    return rc;
}

// Pruning profile (desmo_pruning_profile): library planes + the gathered step operands per chunk of points, GEMM 1 transposed with the
// pruning epilogue, then fixed-order sums of the per-CTA partials.  The term order travels by value (two bytes a term), so the call
// needs no host-to-device copy and stays capturable.
struct PruneOrder {
    uint16_t k[DESMO_MAX_K];
};

// B [steps + 1][mp]: row s = W[order[s - 1]][t] for t < m; row 0 and the columns t >= m are zero
__global__ void __launch_bounds__(256) prune_b_kernel(const float* __restrict__ W, int mld, int m, int mp, int steps,
                                                      const __grid_constant__ PruneOrder ord, float* __restrict__ B) {
    const long long total = (long long)(steps + 1) * mp;
    for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < total; i += (long long)gridDim.x * 256) {
        const int o = (int)(i / mp), t = (int)(i - (long long)o * mp);
        B[i] = (o > 0 && t < m) ? W[(long long)ord.k[o - 1] * mld + t] : 0.0f;
    }
}

// A [steps + 1][rows_c]: row s = the fp32 library value of term order[s - 1] at the chunk's points, b1 + (b2 + b3) of its three planes
// (each addition is exact: the planes are the split of that value); row 0 is zero
__global__ void __launch_bounds__(256) prune_a_kernel(const __nv_bfloat16* __restrict__ Gp, int Kr, long long rows_c, int steps,
                                                      const __grid_constant__ PruneOrder ord, float* __restrict__ A) {
    const long long xl = (long long)blockIdx.x * 256 + threadIdx.x;
    if (xl >= rows_c) return;
    const size_t plane = (size_t)Kr * rows_c;
    for (int o = blockIdx.y; o <= steps; o += gridDim.y) {
        float v = 0.0f;
        if (o > 0) {
            const size_t i = (size_t)ord.k[o - 1] * rows_c + xl;
            v = __bfloat162float(Gp[i]) + (__bfloat162float(Gp[plane + i]) + __bfloat162float(Gp[2 * plane + i]));
        }
        A[(size_t)o * rows_c + xl] = v;
    }
}

// snap[o][t] = sum, in CTA order, of the partials of the gpt CTAs that own snapshot tile t / 128; norm[t] the same for row steps + 1
__global__ void __launch_bounds__(256) prune_snapshots_kernel(const double* __restrict__ part, int tiles_m, int gpt, int steps, int m,
                                                              double* __restrict__ snap, double* __restrict__ norm) {
    const int rows = steps + 2;
    const long long i = (long long)blockIdx.x * 256 + threadIdx.x;
    if (i >= (long long)rows * m) return;
    const int o = (int)(i / m), t = (int)(i - (long long)o * m);
    double s = 0.0;
    for (int k = 0; k < gpt; ++k) s += part[((long long)(t / gp::BM + k * tiles_m) * rows + o) * gp::BM + (t % gp::BM)];
    if (o <= steps) snap[(long long)o * m + t] = s;
    else if (norm) norm[t] = s;
}

// Scratch layout of the pruning profile.  gpt CTAs share each 128-snapshot tile (tiles_m * gpt ~ the SM count), every CTA keeps one
// fp64 partial [steps + 2][128], and chunks of points are a multiple of gpt * 128 so that each CTA gets the same number of tiles.
struct PruneLayout {
    int Kr, mp, tiles_m, gpt;
    long long rows_c;
    size_t o_idx, o_deg, o_gp, o_wp, o_a, o_b, o_part, part_bytes, bytes;
};
size_t pruning_profile_layout(const desmo_shape* s, int T, int K, int steps, int sms, PruneLayout* L) {
    L->Kr = (K + 63) / 64 * 64;  // GEMM 1 reads (K + 63) / 64 k-blocks, as residual_profile_gemm_path
    L->mp = (s->m + 127) / 128 * 128;
    L->tiles_m = L->mp / 128;
    const long long ptiles = s->ld / 128;
    long long gpt = sms / L->tiles_m;
    if (gpt < 1) gpt = 1;
    if (gpt > ptiles) gpt = ptiles;
    L->gpt = (int)gpt;
    const size_t per_point = (size_t)3 * L->Kr * 2 + (size_t)(steps + 1) * 4;
    const long long unit = 128 * gpt;
    long long rc = (long long)(kProfileChunkBytes / per_point) / unit * unit;
    if (rc < unit) rc = unit;
    if (rc > s->ld) rc = s->ld;
    L->rows_c = rc;
    size_t off = 0;
    auto take = [&](size_t bytes) { const size_t o = off; off = align_up_g(off + bytes, 1024); return o; };
    L->o_idx = take((size_t)T * 8);
    L->o_deg = take((size_t)T);
    L->o_gp = take((size_t)3 * L->Kr * rc * 2);
    L->o_wp = take((size_t)3 * L->Kr * L->mp * 2);
    L->o_a = take((size_t)(steps + 1) * rc * 4);
    L->o_b = take((size_t)(steps + 1) * L->mp * 4);
    L->part_bytes = (size_t)L->tiles_m * L->gpt * (steps + 2) * gp::BM * sizeof(double);
    L->o_part = take(L->part_bytes);
    L->bytes = off;
    return off;
}

int pruning_profile_gemm_path(const desmo_shape* s, int T, int K, int Kp, const void* U, int u_dtype, const float* P, const float* phi,
                              const float* omega, const float* W, int steps, const int32_t* order, double* snap, double* norm,
                              cudaStream_t st) {
    using namespace gp;
    int dev = 0, sms = 0;
    DESMO_CUDA(cudaGetDevice(&dev));
    DESMO_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    PruneLayout L;
    pruning_profile_layout(s, T, K, steps, sms, &L);
    PruneOrder ord;
    memset(&ord, 0, sizeof(ord));
    for (int i = 0; i < steps; ++i) ord.k[i] = (uint16_t)order[i];
    uint8_t* scratch = nullptr;
    DESMO_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&scratch), L.bytes, st));
    __nv_bfloat16* Gp = reinterpret_cast<__nv_bfloat16*>(scratch + L.o_gp);
    __nv_bfloat16* Wp = reinterpret_cast<__nv_bfloat16*>(scratch + L.o_wp);
    float* A = reinterpret_cast<float*>(scratch + L.o_a);
    float* B = reinterpret_cast<float*>(scratch + L.o_b);
    double* part = reinterpret_cast<double*>(scratch + L.o_part);
    TermTable tab{scratch + L.o_idx, scratch + L.o_deg};
    const int Kr = L.Kr, mp = L.mp, grid = L.tiles_m * L.gpt;
    const long long rows_c = L.rows_c;
    int rc = check_cuda(cudaMemsetAsync(part, 0, L.part_bytes, st), "cudaMemsetAsync");
    CUtensorMap tmW_mn, tmG_mn;
    if (!rc) {
        term_table_kernel<<<(T + 127) / 128, 128, 0, st>>>(s->r, s->polyorder, T, tab, nullptr, K);
        w_planes_kernel<<<Kr, 256, 0, st>>>(W, nullptr, K, Kr, s->m, s->mld, mp, Wp);
        const long long nb = ((long long)(steps + 1) * mp + 255) / 256;
        prune_b_kernel<<<(unsigned)(nb < 4096 ? nb : 4096), 256, 0, st>>>(W, s->mld, s->m, mp, steps, ord, B);
        rc = check_cuda(cudaGetLastError(), "prune_b_kernel");
    }
    // GEMM 1 transposed: Rec^T[t x p] = W^T G^T; A = W planes (MN-major: t contiguous), B = G planes (MN-major: p contiguous)
    if (!rc && !(rc = make_map(&tmW_mn, Wp, mp, 3LL * Kr, 64))) rc = make_map(&tmG_mn, Gp, rows_c, 3LL * Kr, 64);
    for (long long x0 = 0; x0 < s->ld && !rc; x0 += rows_c) {
        const long long pts = (s->ld - x0 < rows_c) ? s->ld - x0 : rows_c;  // multiple of 128
        const unsigned bx = (unsigned)((rows_c + 255) / 256);
        library_planes_kernel<<<dim3(bx, 64u), 256, 0, st>>>(P, phi, omega, tab, nullptr, s->r, T, K, Kr, s->n, s->ld, x0, rows_c, Gp);
        prune_a_kernel<<<dim3(bx, (unsigned)(steps + 1 < 64 ? steps + 1 : 64)), 256, 0, st>>>(Gp, Kr, rows_c, steps, ord, A);
        if ((rc = check_cuda(cudaGetLastError(), "prune_a_kernel"))) break;
        GemmArgs g{};
        g.U = U; g.loss_part = part; g.prune_a = A; g.prune_b = B; g.steps = steps;
        g.n = s->n; g.ld = s->ld; g.x0 = x0; g.rows_r = rows_c; g.m = s->m; g.mld = s->mld; g.mp = mp; g.K = K; g.Kp = Kp;
        g.tiles_m = L.tiles_m; g.tiles_n = (int)(pts / 128); g.nslice = 1; g.kblocks = (K + 63) / 64; g.kb_per_slice = g.kblocks;
        g.kgroup = 4; g.a_rows = Kr; g.b_rows = Kr; g.first_chunk = 1;
        // at most `grid` CTAs (a multiple of tiles_m): CTA b owns snapshot tile b % tiles_m and partial slot b in every chunk
        rc = u_dtype == DESMO_DTYPE_BF16 ? launch_gemm<true, true, 3, 3, EPI_PRUNE_BF16>(g, tmW_mn, tmG_mn, grid, st)
                                         : launch_gemm<true, true, 3, 3, EPI_PRUNE>(g, tmW_mn, tmG_mn, grid, st);
    }
    if (!rc) {
        const long long total = (long long)(steps + 2) * s->m;
        prune_snapshots_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(part, L.tiles_m, L.gpt, steps, s->m, snap, norm);
        rc = check_cuda(cudaGetLastError(), "prune_snapshots_kernel");
    }
    cudaFreeAsync(scratch, st);
    return rc;
}

size_t pruning_profile_scratch_bytes(const desmo_shape* s, int T, int K, int steps, int sms) {
    PruneLayout L;
    return pruning_profile_layout(s, T, K, steps, sms, &L);
}

// Residual POD (desmo_residual_gram / desmo_residual_modes): per chunk of points, library planes -> GEMM 1 with the residual epilogue
// (EPI_RESID / EPI_RESID_BF16, as the training step) -> the residual's two bf16 planes, then
//   Gram pass:  the Gram GEMM (EPI_GRAM), both operands the R planes read MN-major (snapshots contiguous), upper tiles only, the
//               contraction split into slices as GEMM 4; then a fixed-order reduce of the slice partials into C_R [m][m] and its trace
//   modes pass: GEMM 3 (EPI_D) with the planes of V / sigma in place of W: Psi [k][ld] = (R V^T / sigma)^T
// Points per chunk: the chunk's G and R planes take about kResidChunkBytes.
constexpr size_t kResidChunkBytes = 64u << 20;

struct ResidLayout {
    int Kr, mp, T, tiles, nslice;
    long long rows_c;
    size_t o_idx, o_deg, o_gp, o_wp, o_rp, o_vp, o_lp, o_part, part_bytes, bytes;
};
size_t residual_pod_layout(const desmo_shape* s, int T, int K, int sms, ResidLayout* L) {
    L->Kr = (K + 63) / 64 * 64;  // GEMM 1 reads (K + 63) / 64 k-blocks, as residual_profile_gemm_path
    L->mp = (s->m + 127) / 128 * 128;
    L->T = L->mp / 128;
    L->tiles = L->T * (L->T + 1) / 2;
    const size_t per_point = (size_t)3 * L->Kr * 2 + (size_t)2 * L->mp * 2;
    long long rc = (long long)(kResidChunkBytes / per_point) / 128 * 128;
    if (rc < 128) rc = 128;
    if (rc > s->ld) rc = s->ld;
    L->rows_c = rc;
    // slices of the contraction: enough work items to fill the SMs, fixed for every chunk (at most one slice per k-block of the first)
    int ns = sms / L->tiles;
    if (ns < 1) ns = 1;
    if (ns > kSliceMax) ns = kSliceMax;
    if (ns > (int)(rc / 64)) ns = (int)(rc / 64);
    L->nslice = ns;
    size_t off = 0;
    auto take = [&](size_t bytes) { const size_t o = off; off = align_up_g(off + bytes, 1024); return o; };
    L->o_idx = take((size_t)T * 8);
    L->o_deg = take((size_t)T);
    L->o_gp = take((size_t)3 * L->Kr * rc * 2);
    L->o_wp = take((size_t)3 * L->Kr * L->mp * 2);
    L->o_rp = take((size_t)2 * rc * L->mp * 2);
    L->o_vp = take((size_t)2 * 128 * L->mp * 2);
    L->o_lp = take((size_t)(sms > 0 ? sms : 1) * sizeof(double));
    L->part_bytes = (size_t)ns * L->tiles * gp::BM * gp::BN * sizeof(double);
    L->o_part = take(L->part_bytes);
    L->bytes = off;
    return off;
}

size_t residual_pod_scratch_bytes(const desmo_shape* s, int T, int K, int sms) {
    ResidLayout L;
    return residual_pod_layout(s, T, K, sms, &L);
}

// C[i][j] = sum over the slices, in order, of the partial of the upper element (min(i, j), max(i, j)): C is exactly symmetric
__global__ void __launch_bounds__(256) resid_gram_reduce_kernel(const double* __restrict__ part, int nslice, int tiles, int T, int m,
                                                                float* __restrict__ C) {
    const long long e = (long long)blockIdx.x * 256 + threadIdx.x;
    if (e >= (long long)m * m) return;
    const int i = (int)(e / m), j = (int)(e - (long long)i * m);
    const int a = i < j ? i : j, b = i < j ? j : i;
    const int tm = a / gp::BM, tn = b / gp::BN;
    const long long tile = (long long)tm * T - (long long)tm * (tm - 1) / 2 + (tn - tm);
    const long long off = tile * (gp::BM * gp::BN) + (long long)(b % gp::BN) * gp::BM + (a % gp::BM);
    const long long stride = (long long)tiles * gp::BM * gp::BN;
    double s = 0.0;
    for (int q = 0; q < nslice; ++q) s += part[q * stride + off];
    C[e] = (float)s;
}

// trace = sum_t C_R[t][t] in fp64 (the slice sums of the diagonal, before the fp32 rounding), one block, fixed order
__global__ void __launch_bounds__(256) resid_gram_trace_kernel(const double* __restrict__ part, int nslice, int tiles, int T, int m,
                                                               double* __restrict__ trace) {
    __shared__ double red[256];
    const long long stride = (long long)tiles * gp::BM * gp::BN;
    double acc = 0.0;
    for (int t = threadIdx.x; t < m; t += 256) {
        const int tm = t / gp::BM;
        const long long tile = (long long)tm * T - (long long)tm * (tm - 1) / 2;
        const long long off = tile * (gp::BM * gp::BN) + (long long)(t % gp::BM) * (gp::BM + 1);
        double s = 0.0;
        for (int q = 0; q < nslice; ++q) s += part[q * stride + off];
        acc += s;
    }
    red[threadIdx.x] = acc;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) *trace = red[0];
}

// planes of V / sigma: Vp [2][128][mp], row i = V[i][t] / sigma[i] for i < k, t < m (a zero row when sigma_i = 0), other entries 0
__global__ void __launch_bounds__(256) mode_planes_kernel(const float* __restrict__ V, const float* __restrict__ sigma, int k, int m, int mp,
                                                          __nv_bfloat16* __restrict__ Vp) {
    const int i = blockIdx.x;
    const float sg = i < k ? sigma[i] : 0.0f;
    for (int t = threadIdx.x; t < mp; t += 256) {
        const float w = (i < k && t < m && sg > 0.0f) ? V[(long long)i * m + t] / sg : 0.0f;
        const __nv_bfloat16 b1 = __float2bfloat16_rn(w);
        const __nv_bfloat16 b2 = __float2bfloat16_rn(w - __bfloat162float(b1));
        Vp[(size_t)i * mp + t] = b1;
        Vp[(size_t)(128 + i) * mp + t] = b2;
    }
}

// Shared by both passes: library planes + GEMM 1 (the residual planes) per chunk, then the pass's own GEMM.  V == nullptr: Gram pass.
static int residual_pod_gemm_path(const desmo_shape* s, int T, int K, int Kp, const void* U, int u_dtype, const float* P, const float* phi,
                                  const float* omega, const float* W, float* Cout, double* trace, int k, const float* V, const float* sigma,
                                  float* modes, void* scratch_v, cudaStream_t st) {
    using namespace gp;
    int dev = 0, sms = 0;
    DESMO_CUDA(cudaGetDevice(&dev));
    DESMO_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    ResidLayout L;
    residual_pod_layout(s, T, K, sms, &L);
    uint8_t* scratch = static_cast<uint8_t*>(scratch_v);
    __nv_bfloat16* Gp = reinterpret_cast<__nv_bfloat16*>(scratch + L.o_gp);
    __nv_bfloat16* Wp = reinterpret_cast<__nv_bfloat16*>(scratch + L.o_wp);
    __nv_bfloat16* Rp = reinterpret_cast<__nv_bfloat16*>(scratch + L.o_rp);
    __nv_bfloat16* Vp = reinterpret_cast<__nv_bfloat16*>(scratch + L.o_vp);
    double* lp = reinterpret_cast<double*>(scratch + L.o_lp);
    double* part = reinterpret_cast<double*>(scratch + L.o_part);
    TermTable tab{scratch + L.o_idx, scratch + L.o_deg};
    const int Kr = L.Kr, mp = L.mp;
    const long long rows_c = L.rows_c;
    const bool gram = V == nullptr;
    term_table_kernel<<<(T + 127) / 128, 128, 0, st>>>(s->r, s->polyorder, T, tab, nullptr, K);
    w_planes_kernel<<<Kr, 256, 0, st>>>(W, nullptr, K, Kr, s->m, s->mld, mp, Wp);
    if (!gram) mode_planes_kernel<<<128, 256, 0, st>>>(V, sigma, k, s->m, mp, Vp);
    DESMO_CUDA(cudaGetLastError());
    CUtensorMap tmG_mn, tmW_mn, tmR_mn, tmR_k, tmV_k;
    int rc;
    if ((rc = make_map(&tmG_mn, Gp, rows_c, 3LL * Kr, 64)) || (rc = make_map(&tmW_mn, Wp, mp, 3LL * Kr, 64))) return rc;
    // R planes [2*rows_c rows][mp]: MN-major A and B of the Gram GEMM (as GEMM 4's A), K-major A of GEMM 3
    if ((rc = make_map(&tmR_mn, Rp, mp, 2LL * rows_c, 64)) || (rc = make_map(&tmR_k, Rp, mp, 2LL * rows_c, 128))) return rc;
    if ((rc = make_map(&tmV_k, Vp, mp, 2LL * 128, 128))) return rc;
    bool first = true;
    for (long long x0 = 0; x0 < s->ld; x0 += rows_c, first = false) {
        const long long pts = (s->ld - x0 < rows_c) ? s->ld - x0 : rows_c;  // multiple of 128
        library_planes_kernel<<<dim3((unsigned)((rows_c + 255) / 256), 64u), 256, 0, st>>>(P, phi, omega, tab, nullptr, s->r, T, K, Kr, s->n,
                                                                                          s->ld, x0, rows_c, Gp);
        DESMO_CUDA(cudaGetLastError());
        GemmArgs g{};
        g.U = U; g.Rp = Rp; g.loss_part = lp;
        g.n = s->n; g.ld = s->ld; g.x0 = x0; g.rows_r = rows_c; g.m = s->m; g.mld = s->mld; g.mp = mp; g.K = K; g.Kp = Kp;
        g.first_chunk = 1;
        // GEMM 1, as the training step's: Rec[p x t] = G W, epilogue r = Rec - U -> two bf16 planes of r
        g.tiles_m = (int)(pts / 128); g.tiles_n = mp / 128; g.nslice = 1; g.kblocks = (K + 63) / 64; g.kb_per_slice = g.kblocks; g.kgroup = 4;
        g.a_rows = Kr; g.b_rows = Kr;
        rc = u_dtype == DESMO_DTYPE_BF16 ? launch_gemm<true, true, 3, 3, EPI_RESID_BF16>(g, tmG_mn, tmW_mn, sms, st)
                                         : launch_gemm<true, true, 3, 3, EPI_RESID>(g, tmG_mn, tmW_mn, sms, st);
        if (rc) return rc;
        if (gram) {
            // C_R tiles (tm <= tn) [t1 x t2] = R^T R; A = B = R (MN-major: t contiguous), contraction over the chunk's points in
            // L.nslice slices; chains of 4 k-blocks (48 MMAs) per TMEM accumulator, summed in fp32 RN, then fp64 across the chunks
            g.loss_part = part; g.first_chunk = first ? 1 : 0;
            g.tiles_m = 1; g.tiles_n = L.tiles; g.kblocks = (int)(pts / 64); g.nslice = L.nslice;
            g.kb_per_slice = (g.kblocks + g.nslice - 1) / g.nslice; g.kgroup = 4;
            g.a_rows = (int)rows_c; g.b_rows = (int)rows_c;
            rc = launch_gemm<true, true, 2, 2, EPI_GRAM>(g, tmR_mn, tmR_mn, sms, st);
        } else {
            // GEMM 3, as the training step's: Psi^T[p x mode] = R (V / sigma)^T; A = R (K-major), B = V planes (K-major)
            g.Dacc = modes; g.K = k; g.n_lib16 = (k + 15) / 16 * 16;
            g.tiles_m = (int)(pts / 128); g.tiles_n = 1; g.nslice = 1; g.kblocks = mp / 64; g.kb_per_slice = g.kblocks; g.kgroup = 32;
            g.a_rows = (int)rows_c; g.b_rows = 128;
            rc = launch_gemm<false, false, 2, 2, EPI_D>(g, tmR_k, tmV_k, sms, st);
        }
        if (rc) return rc;
    }
    if (gram) {
        const long long total = (long long)s->m * s->m;
        resid_gram_reduce_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(part, L.nslice, L.tiles, L.T, s->m, Cout);
        resid_gram_trace_kernel<<<1, 256, 0, st>>>(part, L.nslice, L.tiles, L.T, s->m, trace);
        DESMO_CUDA(cudaGetLastError());
    }
    return DESMO_OK;
}

int residual_gram_gemm_path(const desmo_shape* s, int T, int K, int Kp, const void* U, int u_dtype, const float* P, const float* phi,
                            const float* omega, const float* W, float* C, double* trace, void* scratch, cudaStream_t st) {
    return residual_pod_gemm_path(s, T, K, Kp, U, u_dtype, P, phi, omega, W, C, trace, 0, nullptr, nullptr, nullptr, scratch, st);
}

int residual_modes_gemm_path(const desmo_shape* s, int T, int K, int Kp, const void* U, int u_dtype, const float* P, const float* phi,
                             const float* omega, const float* W, int k, const float* V, const float* sigma, float* modes, void* scratch,
                             cudaStream_t st) {
    return residual_pod_gemm_path(s, T, K, Kp, U, u_dtype, P, phi, omega, W, nullptr, nullptr, k, V, sigma, modes, scratch, st);
}

// Backward elimination pass (desmo_elimination_pass): per chunk of points, library planes -> GEMM 1 with the residual epilogue (EPI_RESID
// / EPI_RESID_BF16, as the training step: r's two bf16 planes and sum r^2) -> then
//   GEMM 4 (EPI_E, as the training step): this chunk's slices of F^T = R^T G, added in slice order into the fp64 F [K][mld]
//   the library Gram GEMM (EPI_GRAM): both operands the three G planes read K-major through GEMM 4's B map, upper tiles only, the
//               contraction over the chunk's points split into slices fixed for every chunk, fp64 slice partials accumulated over the
//               chunks; then a fixed-order reduce into the fp64 A [K][K], mirrored.
// Points per chunk: the chunk's G and R planes take about kElimChunkBytes.
constexpr size_t kElimChunkBytes = 64u << 20;

struct ElimLayout {
    int Kr, Kp16, mp, TK, tiles, nslice_g, nslice_e;
    long long rows_c;
    size_t o_idx, o_deg, o_gp, o_wp, o_rp, o_ep, o_lp, o_part, part_bytes, bytes;
};
size_t elimination_layout(const desmo_shape* s, int T, int K, int sms, ElimLayout* L) {
    L->Kr = (K + 127) / 128 * 128;  // GEMM 4 and the Gram GEMM read tiles of 128 library rows
    L->Kp16 = (K + 15) / 16 * 16;
    L->mp = (s->m + 127) / 128 * 128;
    L->TK = L->Kr / 128;
    L->tiles = L->TK * (L->TK + 1) / 2;
    const size_t per_point = (size_t)3 * L->Kr * 2 + (size_t)2 * L->mp * 2;
    long long rc = (long long)(kElimChunkBytes / per_point) / 128 * 128;
    if (rc < 128) rc = 128;
    if (rc > s->ld) rc = s->ld;
    L->rows_c = rc;
    // slices of the two contractions over the points: enough work items to fill the SMs, the same for every chunk
    auto slices = [&](int tiles) {
        int ns = sms / tiles;
        if (ns < 1) ns = 1;
        if (ns > kSliceMax) ns = kSliceMax;
        if (ns > (int)(rc / 64)) ns = (int)(rc / 64);
        return ns;
    };
    L->nslice_g = slices(L->tiles);
    L->nslice_e = slices((L->mp / 128) * L->TK);
    size_t off = 0;
    auto take = [&](size_t bytes) { const size_t o = off; off = align_up_g(off + bytes, 1024); return o; };
    L->o_idx = take((size_t)T * 8);
    L->o_deg = take((size_t)T);
    L->o_gp = take((size_t)3 * L->Kr * rc * 2);
    L->o_wp = take((size_t)3 * L->Kr * L->mp * 2);
    L->o_rp = take((size_t)2 * rc * L->mp * 2);
    L->o_ep = take((size_t)L->nslice_e * L->Kp16 * s->mld * 4);
    L->o_lp = take((size_t)(sms > 0 ? sms : 1) * sizeof(double));
    L->part_bytes = (size_t)L->nslice_g * L->tiles * gp::BM * gp::BN * sizeof(double);
    L->o_part = take(L->part_bytes);
    L->bytes = off;
    return off;
}

size_t elimination_scratch_bytes(const desmo_shape* s, int T, int K, int sms) {
    ElimLayout L;
    return elimination_layout(s, T, K, sms, &L);
}

// F [K][mld] fp64: the first chunk stores, later chunks add, the sum of this chunk's E slices [nslice][Kp16][mld] in slice order
__global__ void __launch_bounds__(256) elim_f_accum_kernel(const float* __restrict__ Ep, int nslice, int K, int Kp16, int mld, int first,
                                                           double* __restrict__ F) {
    const long long e = (long long)blockIdx.x * 256 + threadIdx.x;
    if (e >= (long long)K * mld) return;
    const long long slice = (long long)Kp16 * mld;
    double s = 0.0;
    for (int q = 0; q < nslice; ++q) s += (double)Ep[q * slice + e];
    F[e] = first ? s : F[e] + s;
}

// A[i][j] = sum over the slices, in order, of the partial of the upper element (min(i, j), max(i, j)): A is exactly symmetric.
// Block 0 also writes r2 = the GEMM 1 loss partials summed in CTA order.
__global__ void __launch_bounds__(256) elim_gram_reduce_kernel(const double* __restrict__ part, int nslice, int tiles, int TK, int K,
                                                               const double* __restrict__ lp, int nloss, double* __restrict__ A,
                                                               double* __restrict__ r2) {
    const long long e = (long long)blockIdx.x * 256 + threadIdx.x;
    if (e == 0) {
        double s = 0.0;
        for (int b = 0; b < nloss; ++b) s += lp[b];
        *r2 = s;
    }
    if (e >= (long long)K * K) return;
    const int i = (int)(e / K), j = (int)(e - (long long)i * K);
    const int a = i < j ? i : j, b = i < j ? j : i;
    const int tm = a / gp::BM, tn = b / gp::BN;
    const long long tile = (long long)tm * TK - (long long)tm * (tm - 1) / 2 + (tn - tm);
    const long long off = tile * (gp::BM * gp::BN) + (long long)(b % gp::BN) * gp::BM + (a % gp::BM);
    const long long stride = (long long)tiles * gp::BM * gp::BN;
    double s = 0.0;
    for (int q = 0; q < nslice; ++q) s += part[q * stride + off];
    A[e] = s;
}

int elimination_pass_gemm_path(const desmo_shape* s, int T, int K, const void* U, int u_dtype, const float* P, const float* phi,
                               const float* omega, const float* W, double* A, double* F, double* r2, void* scratch_v, cudaStream_t st) {
    using namespace gp;
    int dev = 0, sms = 0;
    DESMO_CUDA(cudaGetDevice(&dev));
    DESMO_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    ElimLayout L;
    elimination_layout(s, T, K, sms, &L);
    uint8_t* scratch = static_cast<uint8_t*>(scratch_v);
    __nv_bfloat16* Gp = reinterpret_cast<__nv_bfloat16*>(scratch + L.o_gp);
    __nv_bfloat16* Wp = reinterpret_cast<__nv_bfloat16*>(scratch + L.o_wp);
    __nv_bfloat16* Rp = reinterpret_cast<__nv_bfloat16*>(scratch + L.o_rp);
    float* Ep = reinterpret_cast<float*>(scratch + L.o_ep);
    double* lp = reinterpret_cast<double*>(scratch + L.o_lp);
    double* part = reinterpret_cast<double*>(scratch + L.o_part);
    TermTable tab{scratch + L.o_idx, scratch + L.o_deg};
    const int Kr = L.Kr, mp = L.mp;
    const long long rows_c = L.rows_c;
    term_table_kernel<<<(T + 127) / 128, 128, 0, st>>>(s->r, s->polyorder, T, tab, nullptr, K);
    w_planes_kernel<<<Kr, 256, 0, st>>>(W, nullptr, K, Kr, s->m, s->mld, mp, Wp);
    DESMO_CUDA(cudaGetLastError());
    CUtensorMap tmG_mn, tmG_k, tmW_mn, tmR_mn;
    int rc;
    // G planes [3*Kr rows][rows_c]: MN-major A of GEMM 1, K-major B of GEMM 4 and both operands of the Gram GEMM
    if ((rc = make_map(&tmG_mn, Gp, rows_c, 3LL * Kr, 64)) || (rc = make_map(&tmG_k, Gp, rows_c, 3LL * Kr, 128))) return rc;
    if ((rc = make_map(&tmW_mn, Wp, mp, 3LL * Kr, 64)) || (rc = make_map(&tmR_mn, Rp, mp, 2LL * rows_c, 64))) return rc;
    int nloss = 0;
    bool first = true;
    for (long long x0 = 0; x0 < s->ld; x0 += rows_c, first = false) {
        const long long pts = (s->ld - x0 < rows_c) ? s->ld - x0 : rows_c;  // multiple of 128
        library_planes_kernel<<<dim3((unsigned)((rows_c + 255) / 256), 64u), 256, 0, st>>>(P, phi, omega, tab, nullptr, s->r, T, K, Kr, s->n,
                                                                                          s->ld, x0, rows_c, Gp);
        DESMO_CUDA(cudaGetLastError());
        GemmArgs g{};
        g.U = U; g.Rp = Rp; g.Epart = Ep; g.loss_part = lp;
        g.n = s->n; g.ld = s->ld; g.x0 = x0; g.rows_r = rows_c; g.m = s->m; g.mld = s->mld; g.mp = mp; g.K = K; g.Kp = L.Kp16;
        g.n_lib16 = L.Kp16;
        // GEMM 1, as the training step's: Rec[p x t] = G W, epilogue r = Rec - U -> two bf16 planes of r, sum r^2 per CTA over the chunks
        g.first_chunk = first ? 1 : 0;
        g.tiles_m = (int)(pts / 128); g.tiles_n = mp / 128; g.nslice = 1; g.kblocks = (K + 63) / 64; g.kb_per_slice = g.kblocks; g.kgroup = 4;
        g.a_rows = Kr; g.b_rows = Kr;
        rc = u_dtype == DESMO_DTYPE_BF16 ? launch_gemm<true, true, 3, 3, EPI_RESID_BF16>(g, tmG_mn, tmW_mn, sms, st)
                                         : launch_gemm<true, true, 3, 3, EPI_RESID>(g, tmG_mn, tmW_mn, sms, st);
        if (rc) return rc;
        if (first) nloss = g.tiles_m * g.tiles_n < sms ? g.tiles_m * g.tiles_n : sms;  // the first chunk is the largest
        // GEMM 4, as the training step's: E^T[t x lib] = R^T G; A = R (MN-major), B = G (K-major), this chunk's points in slices
        g.first_chunk = 1;
        g.tiles_m = mp / 128; g.tiles_n = L.TK; g.kblocks = (int)(pts / 64); g.nslice = L.nslice_e;
        g.kb_per_slice = (g.kblocks + g.nslice - 1) / g.nslice; g.kgroup = 32;
        g.a_rows = (int)rows_c; g.b_rows = Kr;
        if ((rc = launch_gemm<true, false, 2, 2, EPI_E>(g, tmR_mn, tmG_k, sms, st))) return rc;
        const long long fcount = (long long)K * s->mld;
        elim_f_accum_kernel<<<(unsigned)((fcount + 255) / 256), 256, 0, st>>>(Ep, L.nslice_e, K, L.Kp16, s->mld, first ? 1 : 0, F);
        DESMO_CUDA(cudaGetLastError());
        // Gram GEMM: A tiles (tm <= tn) [k1 x k2] = G^T G; A = B = G (K-major: p contiguous), the six products of GEMM 1, chains of 2
        // k-blocks (48 MMAs) per TMEM accumulator, summed in fp32 RN within a slice, fp64 across slices and chunks
        g.loss_part = part; g.first_chunk = first ? 1 : 0; g.mp = Kr;
        g.tiles_m = 1; g.tiles_n = L.tiles; g.kblocks = (int)(pts / 64); g.nslice = L.nslice_g;
        g.kb_per_slice = (g.kblocks + g.nslice - 1) / g.nslice; g.kgroup = 2;
        g.a_rows = Kr; g.b_rows = Kr;
        if ((rc = launch_gemm<false, false, 3, 3, EPI_GRAM>(g, tmG_k, tmG_k, sms, st))) return rc;
    }
    const long long total = (long long)K * K;
    elim_gram_reduce_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(part, L.nslice_g, L.tiles, L.TK, K, lp, nloss, A, r2);
    DESMO_CUDA(cudaGetLastError());
    return DESMO_OK;
}

int colnorm2_gemm_path(const desmo_shape* s, int T, int K, const float* P, const float* phi, const float* omega, float* out_k, cudaStream_t st) {
    using namespace gp;
    void* scratch = nullptr;
    const size_t bytes = (size_t)T * 9 + 2048;
    DESMO_CUDA(cudaMallocAsync(&scratch, bytes, st));
    TermTable tab{static_cast<uint8_t*>(scratch), static_cast<uint8_t*>(scratch) + align_up_g((size_t)T * 8, 256)};
    term_table_kernel<<<(T + 127) / 128, 128, 0, st>>>(s->r, s->polyorder, T, tab, nullptr, K);
    DESMO_CUDA(cudaMemsetAsync(out_k, 0, sizeof(float) * K, st));
    colnorm2_generic_kernel<<<(unsigned)((s->n + 255) / 256), 256, 0, st>>>(P, phi, omega, tab, s->r, T, K, s->n, s->ld, out_k);
    DESMO_CUDA(cudaGetLastError());
    cudaFreeAsync(scratch, st);
    return DESMO_OK;
}

}  // namespace desmo
