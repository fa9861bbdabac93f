// POD initialisation by the method of snapshots (replaces np.linalg.svd of the n x m data matrix, CYL:197-205):
//   C = U U^T (m x m Gram over mesh points; the one dense contraction)  ->  top-r eigenpairs (lambda_i, v_i) on device
//   ->  POD mode i = X v_i / sqrt(lambda_i), i.e. P[i][x] = sum_t U[t][x] v_i[t] / sigma_i.
// Point-sharded: each rank forms the Gram of its slab, one all-reduce of C, replicated eigensolve, local projection.
#include <algorithm>

#include "common.cuh"

namespace desmo {

// ---------------------------------------------------------------------------------------------------------------
// Gram, FFMA version (the tcgen05 version -- three bf16 planes per fp32 operand -- lives in gram_tc.cu): 64x64 output tile per CTA, split over points.
// ---------------------------------------------------------------------------------------------------------------
constexpr int kGT = 64;   // output tile edge
constexpr int kGX = 32;   // points per smem stage
constexpr int kGP = 68;   // smem pitch

// UT = float or __nv_bfloat16 (snapshots stored in bf16 are widened exactly; the products and sums are the same fp32 FFMAs)
template <class UT>
__global__ void __launch_bounds__(256) gram_fp32_kernel(const UT* __restrict__ U, long long ld, long long n, int m,
                                                        int ntile, long long xchunk, float* __restrict__ C) {
    __shared__ __align__(16) float As[kGX][kGP];
    __shared__ __align__(16) float Bs[kGX][kGP];
    // decode upper-triangular tile pair
    int pair = blockIdx.x, bi = 0;
    while (pair >= ntile - bi) { pair -= ntile - bi; ++bi; }
    const int bj = bi + pair;
    const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
    const long long x0 = (long long)blockIdx.y * xchunk;
    const long long x1 = (x0 + xchunk < n) ? x0 + xchunk : n;
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.0f;
    for (long long xb = x0; xb < x1; xb += kGX) {
        for (int e = tid; e < kGT * kGX; e += 256) {
            const int t = e / kGX, xx = e % kGX;
            const long long x = xb + xx;
            const int ta = bi * kGT + t, tb = bj * kGT + t;
            As[xx][t] = (ta < m && x < x1) ? (float)U[(long long)ta * ld + x] : 0.0f;
            Bs[xx][t] = (tb < m && x < x1) ? (float)U[(long long)tb * ld + x] : 0.0f;
        }
        __syncthreads();
#pragma unroll 8
        for (int xx = 0; xx < kGX; ++xx) {
            const float4 av = *reinterpret_cast<const float4*>(&As[xx][ty * 4]);
            const float4 bv = *reinterpret_cast<const float4*>(&Bs[xx][tx * 4]);
            const float aa[4] = {av.x, av.y, av.z, av.w}, bb[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(aa[i], bb[j], acc[i][j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int ta = bi * kGT + ty * 4 + i, tb = bj * kGT + tx * 4 + j;
            if (ta < m && tb < m) {
                atomicAdd(C + (long long)ta * m + tb, acc[i][j]);
                if (bi != bj) atomicAdd(C + (long long)tb * m + ta, acc[i][j]);
            }
        }
}

int pod_gram_fp32(const desmo_shape* s, const void* U, int u_dtype, float* C, cudaStream_t st) {
    const int m = s->m, ntile = (m + kGT - 1) / kGT;
    const int npairs = ntile * (ntile + 1) / 2;
    DESMO_CUDA(cudaMemsetAsync(C, 0, sizeof(float) * (size_t)m * m, st));
    long long nsplit = (148LL * 8 + npairs - 1) / npairs;
    const long long maxsplit = (s->n + 4095) / 4096;
    if (nsplit > maxsplit) nsplit = maxsplit;
    if (nsplit < 1) nsplit = 1;
    long long xchunk = ((s->n + nsplit - 1) / nsplit + kGX - 1) / kGX * kGX;
    nsplit = (s->n + xchunk - 1) / xchunk;
    if (u_dtype == DESMO_DTYPE_BF16)
        gram_fp32_kernel<<<dim3(npairs, (unsigned)nsplit), 256, 0, st>>>(static_cast<const __nv_bfloat16*>(U), s->ld, s->n, m, ntile, xchunk, C);
    else
        gram_fp32_kernel<<<dim3(npairs, (unsigned)nsplit), 256, 0, st>>>(static_cast<const float*>(U), s->ld, s->n, m, ntile, xchunk, C);
    DESMO_CUDA(cudaGetLastError());
    return DESMO_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// Top-r eigenpairs of the (all-reduced) Gram: block subspace iteration with b = min(r + 8, 16, m) vectors in fp64, CGS2 each
// sweep, Rayleigh-Ritz (cyclic Jacobi on the b x b projection).  After kEigMinIters sweeps, and every kEigCheckEvery sweeps after
// that, a Rayleigh-Ritz pass emits the top r pairs and measures their residuals ||C x_i - theta_i x_i||; the iteration stops once
// every mode above the floor has a residual <= 2^-27 lambda_1, at the latest after a cap of 240 (r <= 8) or 600 sweeps.  The stop is a device
// flag: the launches of the capped loop that follow it return at once, so the solver stays stream-ordered and capturable.
// ---------------------------------------------------------------------------------------------------------------
constexpr int kEigMaxB = 16;
constexpr int kEigMinIters = 120;    // sweeps before the first check: r <= 8 results stay those of the fixed 120-sweep solver
constexpr int kEigCheckEvery = 20;
// Cap.  Every sweep enqueued after convergence still costs two launches that return at once (~1.2 us each on a B200), so the cap
// follows the number of guard vectors: with 8 (r <= 8) a spectrum as flat as sigma_i ~ (i+1)^-0.15 converges within 120 sweeps;
// with 2 (r = 14) it needs ~300.
constexpr int kEigMaxItersSmallR = 240, kEigMaxIters = 600;
constexpr double kEigTol = 0x1p-27;  // residual / lambda_1 (7.5e-9): 2x below the fp32 rounding of C

// workspace head: written by the solver, read by the caller after the stream has passed the eigensolve (include/desmo_b200.h)
struct EigState {
    int32_t iterations;  // sweeps run before the emitted Rayleigh-Ritz pass
    int32_t converged;   // 1: every mode above the floor met the residual bound
    int32_t done;        // stop flag of the capped loop
    int32_t pad;
    double residual;     // max_i ||C x_i - theta_i x_i|| / lambda_1 over the modes above the floor
};
constexpr size_t kEigStateBytes = 256;

__global__ void __launch_bounds__(256) eig_init_kernel(int m, int b, double* V, EigState* st) {
    // deterministic, well-spread start: V[j][t] = cos(pi (j+1)(t+0.5)/m) + small hash noise
    const int t = blockIdx.x * 256 + threadIdx.x;
    if (t == 0) *st = EigState{0, 0, 0, 0, 0.0};
    if (t >= m) return;
    for (int j = 0; j < b; ++j) {
        unsigned h = (unsigned)(t * 2654435761u) ^ (unsigned)((j + 1) * 40503u);
        h ^= h >> 13; h *= 0x5bd1e995u; h ^= h >> 15;
        V[(size_t)j * m + t] = cos(3.141592653589793 * (j + 1) * (t + 0.5) / m) + 1e-3 * ((double)(h & 0xffff) / 65536.0 - 0.5);
    }
}

// Y[j][t] = sum_s C[t][s] V[j][s]   (one warp per row t).  done: the stop flag, NULL for the sweeps before the first check.
__global__ void __launch_bounds__(256) eig_matvec_kernel(int m, int b, const float* __restrict__ C, const double* __restrict__ V,
                                                         double* __restrict__ Y, const int32_t* done) {
    if (done && *done) return;
    const int t = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (t >= m) return;
    double acc[kEigMaxB];
#pragma unroll
    for (int j = 0; j < kEigMaxB; ++j) acc[j] = 0.0;
    for (int s = lane; s < m; s += 32) {
        const double c = (double)C[(size_t)t * m + s];
#pragma unroll
        for (int j = 0; j < kEigMaxB; ++j)
            if (j < b) acc[j] += c * V[(size_t)j * m + s];
    }
#pragma unroll
    for (int j = 0; j < kEigMaxB; ++j)
        if (j < b) {
            const double v = warp_sum(acc[j]);
            if (lane == 0) Y[(size_t)j * m + t] = v;
        }
}

__device__ double block_sum_d(double v, double* sh) {  // blockDim.x == 1024
    v = warp_sum(v);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
    __syncthreads();
    double s = 0.0;
    for (int w = 0; w < 32; ++w) s += sh[w];
    return s;
}

// Classical Gram-Schmidt with re-orthogonalisation (CGS2) of Y (b vectors of length m) -> V, single CTA.  All projections of a
// column onto the previous ones are formed in ONE pass and ONE block reduction (a modified Gram-Schmidt needs one reduction per
// pair: 4x more barriers for the same numerical quality once every column is orthogonalised twice).
__global__ void __launch_bounds__(1024) eig_orth_kernel(int m, int b, const double* __restrict__ Y, double* __restrict__ V,
                                                        const int32_t* done) {
    if (done && *done) return;
    __shared__ double sh[32];
    __shared__ double part[32][kEigMaxB];
    __shared__ double dsum[kEigMaxB];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int j = 0; j < b; ++j) {
        for (int t = threadIdx.x; t < m; t += 1024) V[(size_t)j * m + t] = Y[(size_t)j * m + t];
        __syncthreads();
        for (int pass = 0; pass < 2 && j > 0; ++pass) {
            double d[kEigMaxB];
#pragma unroll
            for (int i = 0; i < kEigMaxB; ++i) d[i] = 0.0;
            for (int t = threadIdx.x; t < m; t += 1024) {
                const double vj = V[(size_t)j * m + t];
#pragma unroll
                for (int i = 0; i < kEigMaxB; ++i)
                    if (i < j) d[i] += V[(size_t)i * m + t] * vj;
            }
#pragma unroll
            for (int i = 0; i < kEigMaxB; ++i)
                if (i < j) {
                    const double w = warp_sum(d[i]);
                    if (lane == 0) part[warp][i] = w;
                }
            __syncthreads();
            if (threadIdx.x < j) {
                double acc = 0.0;
                for (int w = 0; w < 32; ++w) acc += part[w][threadIdx.x];
                dsum[threadIdx.x] = acc;
            }
            __syncthreads();
            for (int t = threadIdx.x; t < m; t += 1024) {
                double v = V[(size_t)j * m + t];
                for (int i = 0; i < j; ++i) v -= dsum[i] * V[(size_t)i * m + t];
                V[(size_t)j * m + t] = v;
            }
            __syncthreads();
        }
        double nn = 0.0;
        for (int t = threadIdx.x; t < m; t += 1024) nn += V[(size_t)j * m + t] * V[(size_t)j * m + t];
        nn = block_sum_d(nn, sh);
        const double inv = (nn > 0.0) ? rsqrt(nn) : 0.0;
        for (int t = threadIdx.x; t < m; t += 1024) V[(size_t)j * m + t] *= inv;
        __syncthreads();
    }
}

// Rayleigh-Ritz: H = V^T (C V) = V^T Y (b x b), Jacobi eigen-decomposition, rotate, sort, sign-normalise, emit top r, and the
// residuals ||Y q_i - theta_i V q_i|| = ||C x_i - theta_i x_i|| of the emitted pairs.  Floor: a Ritz value theta_i <= 2^-23 trace(C)
// is at the rounding level of the fp32 Gram (its eigenvector is noise); it is emitted as sigma_i = 0 and left out of the stop test.
__global__ void __launch_bounds__(1024) eig_ritz_kernel(int m, int b, int r, const float* __restrict__ C, const double* __restrict__ V,
                                                        const double* __restrict__ Y, float* __restrict__ Vout, float* __restrict__ sigma,
                                                        EigState* __restrict__ state, int iteration, int last) {
    if (state->done) return;
    __shared__ double sh[32];
    __shared__ double H[kEigMaxB][kEigMaxB], Q[kEigMaxB][kEigMaxB];
    __shared__ int order[kEigMaxB];
    for (int i = 0; i < b; ++i)
        for (int j = i; j < b; ++j) {
            double d = 0.0;
            for (int t = threadIdx.x; t < m; t += 1024) d += V[(size_t)i * m + t] * Y[(size_t)j * m + t];
            d = block_sum_d(d, sh);
            if (threadIdx.x == 0) { H[i][j] = d; H[j][i] = d; }
        }
    double trace = 0.0;
    for (int t = threadIdx.x; t < m; t += 1024) trace += (double)C[(size_t)t * m + t];
    trace = block_sum_d(trace, sh);
    __syncthreads();
    if (threadIdx.x < 32) {
        // cyclic Jacobi, one warp: every lane derives the same rotation, lane k updates row / column k (the serial sweep's arithmetic)
        const int k = threadIdx.x;
        if (k < b)
            for (int j = 0; j < b; ++j) Q[k][j] = (k == j) ? 1.0 : 0.0;
        __syncwarp();
        for (int sweep = 0; sweep < 30; ++sweep) {
            double off = 0.0;
            for (int p = 0; p < b; ++p)
                for (int q = p + 1; q < b; ++q) off += H[p][q] * H[p][q];
            if (off < 1e-300) break;
            for (int p = 0; p < b; ++p)
                for (int q = p + 1; q < b; ++q) {
                    if (fabs(H[p][q]) < 1e-300) continue;
                    const double theta = (H[q][q] - H[p][p]) / (2.0 * H[p][q]);
                    const double tt = (theta >= 0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
                    const double c = 1.0 / sqrt(tt * tt + 1.0), s2 = tt * c;
                    __syncwarp();
                    if (k < b) {
                        const double hkp = H[k][p], hkq = H[k][q];
                        H[k][p] = c * hkp - s2 * hkq;
                        H[k][q] = s2 * hkp + c * hkq;
                    }
                    __syncwarp();
                    if (k < b) {
                        const double hpk = H[p][k], hqk = H[q][k];
                        H[p][k] = c * hpk - s2 * hqk;
                        H[q][k] = s2 * hpk + c * hqk;
                        const double qkp = Q[k][p], qkq = Q[k][q];
                        Q[k][p] = c * qkp - s2 * qkq;
                        Q[k][q] = s2 * qkp + c * qkq;
                    }
                    __syncwarp();
                }
        }
        if (k == 0) {
            for (int i = 0; i < b; ++i) order[i] = i;
            for (int i = 0; i < b; ++i)
                for (int j = i + 1; j < b; ++j)
                    if (H[order[j]][order[j]] > H[order[i]][order[i]]) { const int tmp = order[i]; order[i] = order[j]; order[j] = tmp; }
        }
    }
    __syncthreads();
    const double lam1 = H[order[0]][order[0]], floor_lam = 0x1p-23 * trace;
    double worst = 0.0;
    for (int i = 0; i < r; ++i) {
        const int col = order[i];
        const double th = H[col][col];
        // ritz vector = sum_j Q[j][col] V[j]; find the largest-|.| entry for the sign convention
        double best = 0.0, res2 = 0.0;
        for (int t = threadIdx.x; t < m; t += 1024) {
            double v = 0.0, cv = 0.0;
            for (int j = 0; j < b; ++j) {
                v += Q[j][col] * V[(size_t)j * m + t];
                cv += Q[j][col] * Y[(size_t)j * m + t];
            }
            if (fabs(v) > fabs(best)) best = v;
            res2 += (cv - th * v) * (cv - th * v);
        }
        res2 = block_sum_d(res2, sh);
        // block arg-max of |best|
        __syncthreads();
        double cand = best;
        for (int o = 16; o > 0; o >>= 1) {
            const double other = __shfl_xor_sync(0xffffffffu, cand, o);
            if (fabs(other) > fabs(cand) || (fabs(other) == fabs(cand) && other > cand)) cand = other;
        }
        if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = cand;
        __syncthreads();
        double top = sh[0];
        for (int w = 1; w < 32; ++w)
            if (fabs(sh[w]) > fabs(top) || (fabs(sh[w]) == fabs(top) && sh[w] > top)) top = sh[w];
        const double flip = (top < 0.0) ? -1.0 : 1.0;
        for (int t = threadIdx.x; t < m; t += 1024) {
            double v = 0.0;
            for (int j = 0; j < b; ++j) v += Q[j][col] * V[(size_t)j * m + t];
            Vout[(size_t)i * m + t] = (float)(flip * v);
        }
        const bool floored = !(th > floor_lam);
        if (!floored) worst = fmax(worst, sqrt(res2) / lam1);
        if (threadIdx.x == 0) sigma[i] = floored ? 0.0f : (float)sqrt(th);
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        const int ok = worst <= kEigTol;
        state->iterations = iteration;
        state->converged = ok;
        state->residual = worst;
        state->done = ok || last;
    }
}

int pod_eig(int m, int r, const float* C, float* V, float* sigma, void* workspace, size_t workspace_bytes, cudaStream_t st) {
    if (r > kEigMaxB - 2) {
        set_error("pod_eig: r=%d exceeds the on-device eigensolver's limit r <= %d", r, kEigMaxB - 2);
        return DESMO_ERR_UNSUPPORTED;
    }
    if (r > m) { set_error("pod_eig: r=%d modes of an m=%d Gram", r, m); return DESMO_ERR_ARG; }
    const int b = std::min(std::min(r + 8, kEigMaxB), m);
    const size_t need = kEigStateBytes + 2 * sizeof(double) * (size_t)b * m;
    if (workspace_bytes < need) { set_error("pod_eig: workspace too small (%zu < %zu)", workspace_bytes, need); return DESMO_ERR_ARG; }
    EigState* state = static_cast<EigState*>(workspace);
    const int32_t* done = &state->done;
    double* Vd = reinterpret_cast<double*>(static_cast<char*>(workspace) + kEigStateBytes);
    double* Yd = Vd + (size_t)b * m;
    eig_init_kernel<<<(m + 255) / 256, 256, 0, st>>>(m, b, Yd, state);
    eig_orth_kernel<<<1, 1024, 0, st>>>(m, b, Yd, Vd, nullptr);
    const int max_iters = r <= 8 ? kEigMaxItersSmallR : kEigMaxIters;
    for (int it = 0;; ++it) {
        const bool checked = it >= kEigMinIters;
        eig_matvec_kernel<<<(m + 7) / 8, 256, 0, st>>>(m, b, C, Vd, Yd, checked ? done : nullptr);
        if (checked && (it - kEigMinIters) % kEigCheckEvery == 0) {
            const int last = it >= max_iters;
            eig_ritz_kernel<<<1, 1024, 0, st>>>(m, b, r, C, Vd, Yd, V, sigma, state, it, last);
            if (last) break;
        }
        eig_orth_kernel<<<1, 1024, 0, st>>>(m, b, Yd, Vd, checked ? done : nullptr);
    }
    DESMO_CUDA(cudaGetLastError());
    return DESMO_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// Back-projection: P[i][x] = sum_t U[t][x] V[i][t] / sigma_i   (HBM-bound; one pass over U per group of kMaxR modes, the groups
// are blockIdx.y; a floored mode, sigma_i = 0, gets a zero row)
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ float4 ldg_u4(const float* U, long long t, long long ld, long long xv) {
    return __ldg(reinterpret_cast<const float4*>(U + t * ld) + xv);
}
__device__ __forceinline__ float4 ldg_u4(const __nv_bfloat16* U, long long t, long long ld, long long xv) {  // one 8-byte load
    const uint2 q = __ldg(reinterpret_cast<const uint2*>(U + t * ld) + xv);
    return make_float4(__uint_as_float(q.x << 16), __uint_as_float(q.x & 0xffff0000u), __uint_as_float(q.y << 16),
                       __uint_as_float(q.y & 0xffff0000u));
}

template <class UT>
__global__ void __launch_bounds__(256) pod_project_kernel(const UT* __restrict__ U, long long ld, long long n, int m, int r,
                                                          const float* __restrict__ V, const float* __restrict__ sigma,
                                                          float* __restrict__ P) {
    extern __shared__ float Vs[];  // [m][kMaxR]: modes g0 .. g0 + kMaxR - 1
    const int g0 = blockIdx.y * kMaxR;
    V += (size_t)g0 * m;
    sigma += g0;
    P += (long long)g0 * ld;
    r -= g0;
    for (int e = threadIdx.x; e < m * kMaxR; e += 256) {
        const int t = e / kMaxR, i = e % kMaxR;
        Vs[e] = (i < r) ? V[(size_t)i * m + t] : 0.0f;
    }
    __syncthreads();
    const long long nvec = ld / 4;
    for (long long xv = (long long)blockIdx.x * 256 + threadIdx.x; xv < nvec; xv += (long long)gridDim.x * 256) {
        float acc[kMaxR][4];
#pragma unroll
        for (int i = 0; i < kMaxR; ++i) acc[i][0] = acc[i][1] = acc[i][2] = acc[i][3] = 0.0f;
#pragma unroll 4
        for (int t = 0; t < m; ++t) {
            const float4 u = ldg_u4(U, t, ld, xv);
            const float4 v0 = *reinterpret_cast<const float4*>(Vs + t * kMaxR);
            const float4 v1 = *reinterpret_cast<const float4*>(Vs + t * kMaxR + 4);
            const float vv[8] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w};
#pragma unroll
            for (int i = 0; i < kMaxR; ++i) {
                acc[i][0] = fmaf(u.x, vv[i], acc[i][0]);
                acc[i][1] = fmaf(u.y, vv[i], acc[i][1]);
                acc[i][2] = fmaf(u.z, vv[i], acc[i][2]);
                acc[i][3] = fmaf(u.w, vv[i], acc[i][3]);
            }
        }
#pragma unroll
        for (int i = 0; i < kMaxR; ++i)
            if (i < r) {
                const float inv = sigma[i] > 0.0f ? 1.0f / sigma[i] : 0.0f;
                const long long x = xv * 4;
                float4 o;
                o.x = (x + 0 < n) ? acc[i][0] * inv : 0.0f;
                o.y = (x + 1 < n) ? acc[i][1] * inv : 0.0f;
                o.z = (x + 2 < n) ? acc[i][2] * inv : 0.0f;
                o.w = (x + 3 < n) ? acc[i][3] * inv : 0.0f;
                *reinterpret_cast<float4*>(P + (long long)i * ld + x) = o;
            }
    }
}

template <class UT>
static int launch_project(const desmo_shape* s, const UT* U, const float* V, const float* sigma, float* P, cudaStream_t st) {
    const size_t smem = sizeof(float) * (size_t)s->m * kMaxR;
    DESMO_CUDA(cudaFuncSetAttribute(pod_project_kernel<UT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    long long g = (s->ld / 4 + 255) / 256;
    if (g > 148 * 4) g = 148 * 4;
    const unsigned groups = (unsigned)((s->r + kMaxR - 1) / kMaxR);
    pod_project_kernel<UT><<<dim3((unsigned)g, groups), 256, smem, st>>>(U, s->ld, s->n, s->m, s->r, V, sigma, P);
    return DESMO_OK;
}

int pod_project(const desmo_shape* s, const void* U, int u_dtype, const float* V, const float* sigma, float* P, cudaStream_t st) {
    const int rc = u_dtype == DESMO_DTYPE_BF16 ? launch_project(s, static_cast<const __nv_bfloat16*>(U), V, sigma, P, st)
                                               : launch_project(s, static_cast<const float*>(U), V, sigma, P, st);
    if (rc) return rc;
    DESMO_CUDA(cudaGetLastError());
    return DESMO_OK;
}

}  // namespace desmo
