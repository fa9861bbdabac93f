// POD Gram matrix C = U U^T (m x m, the one genuinely dense contraction of the path; replaces the O(n m^2) part of
// np.linalg.svd, CYL:199) on the 5th-gen tensor cores: tcgen05.mma kind::f16 with the fp32 snapshots split on the fly into three
// bf16 planes (six products kept -> fp32-class accuracy, like the fused kernel).
//
// A CTA owns one 128 x 128 tile (bi <= bj) of C and one range of mesh points; it walks the range in chunks of 64 points:
//   converter warps (4..11): coalesced 128-bit loads of U[t][x..x+63] for the tile's row blocks (registers, one chunk ahead),
//                            fp32 -> 3 x bf16, 128B-swizzled K-major planes in shared memory (double-buffered);
//   warp 1 (one elected thread): 24 MMAs per chunk (6 plane pairs x 4 k-steps of 16 points), accumulator in TMEM (128 columns);
//   end: TMEM -> registers -> atomicAdd into C (and the mirrored tile).
// Both operands are K-major because the time-major layout keeps mesh points contiguous.
// bf16 snapshots (gram_tc_kernel<true>): the rows already are bf16 MMA operands, so the converters copy them into plane 1 as they are
// and the issuer runs only the plane-1 x plane-1 products (4 MMAs per chunk), in the same k-step order and with the same FLUSH
// cadence: for such data the fp32 kernel's planes 2 and 3 are exactly zero, so the result equals the fp32 Gram of U_q.float().
#include <cuda_bf16.h>

#include "common.cuh"
#include "tcgen05.cuh"

namespace desmo {
namespace gram {
using namespace ptx;

constexpr int BM = 128;            // rows (snapshots) per tile edge
constexpr int BK = 64;             // mesh points per chunk (= one 128 B swizzled row of bf16)
constexpr int CONV_WARPS = 8;
constexpr int PACE = 32;           // chunks between pacing points of the CTAs that stream the same range of mesh points (see the kernel)
constexpr int FLUSH = 16;          // chunks between accumulator flushes: the tensor core truncates when it adds into the fp32
                                   // accumulator (bias ~1e-8 per MMA), so chains are kept to 16 x 24 MMAs and summed in fp32 RN outside
constexpr int THREADS = 128 + CONV_WARPS * 32;
constexpr uint32_t PLANE = BM * 128;                 // one bf16 plane of one operand: [128 rows][128 B]
constexpr uint32_t OPERAND = 3 * PLANE;              // 49152
constexpr uint32_t STAGE = 2 * OPERAND;              // A planes + B planes
constexpr uint32_t SMEM_BYTES = 2 * STAGE + 1024;    // two stages + alignment slack

// Every wait carries a watchdog: a wait still open after ~10 s (by %globaltimer, read only once the first try has failed) traps,
// so a protocol error fails the launch instead of hanging the GPU.  The 10 ms suspend hint parks the waiting warps.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    if (mbar_try_wait(bar, parity, 0x989680u)) return;
    const unsigned long long t0 = globaltimer_ns();
    while (!mbar_try_wait(bar, parity, 0x989680u))
        if (globaltimer_ns() - t0 > 10000000000ull) __trap();
}
// volatile: keeps the next chunk's loads BELOW the current chunk's split + stores (hoisted, they double the live registers and spill)
__device__ __forceinline__ float4 ldg_nc_v4(const float4* p) {
    float4 v;
    asm volatile("ld.global.nc.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
    return v;
}
__device__ __forceinline__ uint4 ldg_nc_u4(const uint4* p) {
    uint4 v;
    asm volatile("ld.global.nc.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
    return v;
}
__device__ __forceinline__ void split3_pair(float x0, float x1, uint32_t& w1, uint32_t& w2, uint32_t& w3) {
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(w1) : "f"(x1), "f"(x0));
    const float e0 = x0 - __uint_as_float(w1 << 16), e1 = x1 - __uint_as_float(w1 & 0xffff0000u);
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(w2) : "f"(e1), "f"(e0));
    const float f0 = e0 - __uint_as_float(w2 << 16), f1 = e1 - __uint_as_float(w2 & 0xffff0000u);
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(w3) : "f"(f1), "f"(f0));
}

template <bool kU16>
__global__ void __launch_bounds__(THREADS, 1) gram_tc_kernel(const void* __restrict__ Uv, long long ld, int m, int ntile, long long xchunk,
                                                             long long xtotal, float* __restrict__ C, float* __restrict__ part,
                                                             unsigned* __restrict__ pace) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bars[8];
    __shared__ uint32_t tmem_base_s;
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    const uint32_t sbase = smem_u32(smem);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    enum { FULL0 = 0, FULL1, EMPTY0, EMPTY1, ACC_FULL, ACC_EMPTY };
    auto bar = [&](int i) { return smem_u32(&bars[i]); };
    const float* __restrict__ U = static_cast<const float*>(Uv);
    const __nv_bfloat16* __restrict__ U16 = static_cast<const __nv_bfloat16*>(Uv);

    int pair = blockIdx.x, bi = 0;
    while (pair >= ntile - bi) { pair -= ntile - bi; ++bi; }
    const int bj = bi + pair;
    const bool diag = (bi == bj);
    const long long x0 = (long long)blockIdx.y * xchunk;
    const long long x1 = (x0 + xchunk < xtotal) ? x0 + xchunk : xtotal;
    const int nchunks = (int)((x1 - x0 + BK - 1) / BK);

    if (tid == 32) {
        mbar_init(bar(FULL0), CONV_WARPS * 32); mbar_init(bar(FULL1), CONV_WARPS * 32);
        mbar_init(bar(EMPTY0), 1); mbar_init(bar(EMPTY1), 1); mbar_init(bar(ACC_FULL), 1); mbar_init(bar(ACC_EMPTY), CONV_WARPS * 32);
        fence_mbar_init();
    }
    if (warp == 2) tmem_alloc<128>(smem_u32(&tmem_base_s));
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_base_s;

    if (warp == 1) {
        if (elect_one_sync()) {
            constexpr uint32_t idesc = make_idesc_bf16(BM, BM, 0, 0);  // K-major both
            uint32_t acc = 0;
            for (int c = 0; c < nchunks; ++c) {
                const int st = c & 1;
                if (c % FLUSH == 0) {
                    if (c > 0) mbar_wait(bar(ACC_EMPTY), ((c / FLUSH) - 1) & 1);  // converters drained the accumulator tile
                    acc = 0;
                }
                mbar_wait(bar(FULL0 + st), (c >> 1) & 1);
                tc_fence_after();
                const uint32_t a_lo = ((sbase + st * STAGE) >> 4) | (1u << 16);
                const uint32_t b_lo = diag ? a_lo : (((sbase + st * STAGE + OPERAND) >> 4) | (1u << 16));
#define GRAM_PAIR(PA, PB)                                                                                                   \
    _Pragma("unroll") for (int ks = 0; ks < BK / 16; ++ks) {                                                                 \
        mma_bf16(tmem, desc_from(a_lo + ((PA * PLANE + ks * 32) >> 4), kDescHi),                                             \
                 desc_from(b_lo + ((PB * PLANE + ks * 32) >> 4), kDescHi), idesc, acc);                                      \
        acc = 1;                                                                                                             \
    }
                if constexpr (kU16) {
                    GRAM_PAIR(0, 0)
                } else {
                    GRAM_PAIR(2, 0) GRAM_PAIR(0, 2) GRAM_PAIR(1, 1) GRAM_PAIR(1, 0) GRAM_PAIR(0, 1) GRAM_PAIR(0, 0)
                }
#undef GRAM_PAIR
                umma_commit(bar(EMPTY0 + st));
                if ((c + 1) % FLUSH == 0 || c == nchunks - 1) umma_commit(bar(ACC_FULL));
            }
        }
    } else if (warp >= 4) {
        // ---------------- converters: 1024 (row, 8-point group) items per operand and chunk, 4 per thread; lanes 0-7 of a warp
        //                  cover the 256 contiguous bytes of one row, so every warp-level load is four full 256 B segments ----------------
        const int ct = tid - 128;            // 0..255
        float4 ra[8], rb[8];
        uint4 qa[4], qb[4];  // bf16: one 16 B load = the 8 points of an item
        auto load_chunk = [&](int c) {
            const long long xo = x0 + (long long)c * BK;
            if constexpr (kU16) {
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const int idx = k * 256 + ct, row = idx >> 3, g8 = idx & 7;
                    const long long x = xo + g8 * 8;
                    const int ta = bi * BM + row, tb = bj * BM + row;
                    const uint4 z = make_uint4(0u, 0u, 0u, 0u);
                    qa[k] = (ta < m && x < x1) ? ldg_nc_u4(reinterpret_cast<const uint4*>(U16 + (long long)ta * ld + x)) : z;
                    if (!diag) qb[k] = (tb < m && x < x1) ? ldg_nc_u4(reinterpret_cast<const uint4*>(U16 + (long long)tb * ld + x)) : z;
                }
                return;
            }
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int idx = k * 256 + ct, row = idx >> 3, g8 = idx & 7;
                const long long x = xo + g8 * 8;
                const int ta = bi * BM + row, tb = bj * BM + row;
                const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
                const float4* qa = reinterpret_cast<const float4*>(U + (long long)ta * ld + x);
                const bool va = ta < m && x < x1;
                ra[2 * k] = va ? ldg_nc_v4(qa) : z;
                ra[2 * k + 1] = va ? ldg_nc_v4(qa + 1) : z;
                if (!diag) {
                    const float4* qb = reinterpret_cast<const float4*>(U + (long long)tb * ld + x);
                    const bool vb = tb < m && x < x1;
                    rb[2 * k] = vb ? ldg_nc_v4(qb) : z;
                    rb[2 * k + 1] = vb ? ldg_nc_v4(qb + 1) : z;
                }
            }
        };
        auto store_planes = [&](uint32_t base, const float4 (&r)[8]) {
            // row `row` of the operand, 16 B chunk g8 (8 points), 128B swizzle; a warp writes four whole 128 B rows per plane
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int idx = k * 256 + ct, row = idx >> 3, g8 = idx & 7;
                uint32_t w1[4], w2[4], w3[4];
                const float4 lo = r[2 * k], hi = r[2 * k + 1];
                split3_pair(lo.x, lo.y, w1[0], w2[0], w3[0]);
                split3_pair(lo.z, lo.w, w1[1], w2[1], w3[1]);
                split3_pair(hi.x, hi.y, w1[2], w2[2], w3[2]);
                split3_pair(hi.z, hi.w, w1[3], w2[3], w3[3]);
                const uint32_t off = row * 128 + ((uint32_t)(g8 ^ (row & 7)) << 4);
                st_shared_v4(base + off, w1[0], w1[1], w1[2], w1[3]);
                st_shared_v4(base + PLANE + off, w2[0], w2[1], w2[2], w2[3]);
                st_shared_v4(base + 2 * PLANE + off, w3[0], w3[1], w3[2], w3[3]);
            }
        };
        auto store_plane16 = [&](uint32_t base, const uint4 (&q)[4]) {  // same rows and swizzle, plane 1 only
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int idx = k * 256 + ct, row = idx >> 3, g8 = idx & 7;
                const uint32_t off = row * 128 + ((uint32_t)(g8 ^ (row & 7)) << 4);
                st_shared_v4(base + off, q[k].x, q[k].y, q[k].z, q[k].w);
            }
        };
        const int q = warp & 3, hcol = (warp - 4) >> 2;
        float* mypart = part + (long long)(blockIdx.y * gridDim.x + blockIdx.x) * (BM * BM);  // [col][row]: lanes -> consecutive rows
        if (nchunks > 0) load_chunk(0);
        for (int c = 0; c < nchunks; ++c) {
            const int st = c & 1;
            if (c > 0 && c % PACE == 0) {
                // Pacing: the gridDim.x tiles of one point range read the same rows of U (every 128-row block is an operand of
                // several tiles); they only share them through L2 while they stay within an L2-sized window of each other, and left
                // alone they drift apart (ncu: 25 GB of DRAM reads for 12.6 GB of data).  Every PACE chunks (a window of PACE * 64
                // points x m rows x 4 ranges = 33 MB) a CTA announces itself and waits -- briefly, with a time limit, so that it
                // is a hint and never a deadlock -- until the others of its range have arrived.
                if (tid == 128) {
                    const unsigned target = (unsigned)gridDim.x * (unsigned)(c / PACE);
                    __threadfence();
                    atomicAdd(pace + blockIdx.y, 1u);
                    const long long t0 = clock64();
                    while (*reinterpret_cast<volatile unsigned*>(pace + blockIdx.y) < target && clock64() - t0 < 40000) __nanosleep(100);
                }
                asm volatile("bar.sync 1, %0;" ::"n"(CONV_WARPS * 32) : "memory");
            }
            if (c >= 2) mbar_wait(bar(EMPTY0 + st), ((c >> 1) - 1) & 1);
            if constexpr (kU16) {
                store_plane16(sbase + st * STAGE, qa);
                if (!diag) store_plane16(sbase + st * STAGE + OPERAND, qb);
            } else {
                store_planes(sbase + st * STAGE, ra);
                if (!diag) store_planes(sbase + st * STAGE + OPERAND, rb);
            }
            if (c + 1 < nchunks) load_chunk(c + 1);  // next chunk's loads fly while this chunk's MMAs run
            fence_async_smem();
            mbar_arrive(bar(FULL0 + st));
            if ((c + 1) % FLUSH == 0 || c == nchunks - 1) {
                // ---- drain the accumulator tile: partial += TMEM (fp32 RN); the last drain goes to C (and its mirror) ----
                const int f = c / FLUSH;
                mbar_wait(bar(ACC_FULL), f & 1);
                tc_fence_after();
#pragma unroll
                for (int cc = 0; cc < 4; ++cc) {
                    uint32_t v[16];
                    float old[16];
                    float* const pp = mypart + (hcol * 64 + cc * 16) * BM + q * 32 + lane;
                    // the 16 partial sums first (independent L2 loads in flight together; one by one they cost a full L2 round trip each)
#pragma unroll
                    for (int j = 0; j < 16; ++j) old[j] = (f == 0) ? 0.0f : __ldcg(pp + j * BM);
                    tmem_ld16(tmem + ((uint32_t)(q * 32) << 16) + hcol * 64 + cc * 16, v);
                    tmem_ld_wait();
#pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        __stcg(pp + j * BM, old[j] + __uint_as_float(v[j]));  // the per-CTA partial tile; summed in a fixed order below
                    }
                }
                tc_fence_before();
                mbar_arrive(bar(ACC_EMPTY));
            }
        }
        tc_fence_before();
    }
    __syncthreads();
    if (warp == 2) {
        tc_fence_after();
        tmem_dealloc<128>(tmem);
    }
}

// C (and its mirror) = sum over the point ranges of the per-CTA partial tiles, in a fixed order: the Gram matrix, and with it the POD
// modes, are bit-reproducible from run to run (atomics into C were not).
__global__ void __launch_bounds__(256) gram_reduce_kernel(const float* __restrict__ part, int npairs, int nsplit, int m, int ntile,
                                                          float* __restrict__ C) {
    int pair = blockIdx.x, bi = 0;
    while (pair >= ntile - bi) { pair -= ntile - bi; ++bi; }
    const int bj = bi + pair;
    for (int e = threadIdx.x; e < BM * BM; e += 256) {
        const int col = e / BM, row = e % BM;  // partial tiles are [col][row]
        float s = 0.0f;
        for (int y = 0; y < nsplit; ++y) s += __ldg(part + ((long long)y * npairs + blockIdx.x) * (BM * BM) + e);
        const int trow = bi * BM + row, tcol = bj * BM + col;
        if (trow < m && tcol < m) {
            C[(long long)trow * m + tcol] = s;
            if (bi != bj) C[(long long)tcol * m + trow] = s;
        }
    }
}

}  // namespace gram

int pod_gram_tc(const desmo_shape* s, const void* U, int u_dtype, float* C, void* workspace, cudaStream_t st) {
    float* part = static_cast<float*>(workspace);  // [SMs][128*128]
    using namespace gram;
    const int m = s->m, ntile = (m + BM - 1) / BM;
    const int npairs = ntile * (ntile + 1) / 2;
    if (npairs > 4096 || s->ld % 4 != 0) return DESMO_ERR_UNSUPPORTED;
    int dev = 0, sms = 0;
    DESMO_CUDA(cudaGetDevice(&dev));
    DESMO_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    DESMO_CUDA(cudaMemsetAsync(C, 0, sizeof(float) * (size_t)m * m, st));
    const long long xtotal = (s->n + BK - 1) / BK * BK <= s->ld ? (s->n + BK - 1) / BK * BK : s->ld;  // padded columns hold zeros
    long long nsplit = sms / npairs;
    if (nsplit < 1) nsplit = 1;
    const long long maxsplit = (xtotal + 4 * BK - 1) / (4 * BK);
    if (nsplit > maxsplit) nsplit = maxsplit;
    long long xchunk = ((xtotal + nsplit - 1) / nsplit + BK - 1) / BK * BK;
    nsplit = (xtotal + xchunk - 1) / xchunk;
    const bool u16 = u_dtype == DESMO_DTYPE_BF16;
    DESMO_CUDA(cudaFuncSetAttribute(u16 ? gram_tc_kernel<true> : gram_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int)SMEM_BYTES));
    if ((long long)npairs * nsplit > sms || nsplit > 256) return DESMO_ERR_UNSUPPORTED;  // one partial tile per SM in the workspace
    unsigned* pace = reinterpret_cast<unsigned*>(part + (size_t)sms * BM * BM);            // pacing counters, one per point range
    DESMO_CUDA(cudaMemsetAsync(pace, 0, 1024, st));
    if (u16) gram_tc_kernel<true><<<dim3(npairs, (unsigned)nsplit), THREADS, SMEM_BYTES, st>>>(U, s->ld, m, ntile, xchunk, xtotal, C, part, pace);
    else gram_tc_kernel<false><<<dim3(npairs, (unsigned)nsplit), THREADS, SMEM_BYTES, st>>>(U, s->ld, m, ntile, xchunk, xtotal, C, part, pace);
    DESMO_CUDA(cudaGetLastError());
    gram_reduce_kernel<<<npairs, 256, 0, st>>>(part, npairs, (int)nsplit, m, ntile, C);
    DESMO_CUDA(cudaGetLastError());
    return DESMO_OK;
}

}  // namespace desmo
