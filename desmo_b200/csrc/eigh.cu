// Dense symmetric eigensolver for the POD Gram (desmo_pod_eigh): every eigenvalue of C and the top-r eigenvectors, in fp64, in a
// time fixed by m and an accuracy that does not depend on the spectrum (the subspace iteration of pod.cu converges at the rate of
// lambda_{b+1} / lambda_r).  LAPACK dsyevx structure:
//   1. tridiagonalise  A = double(C) = Q T Q^T by Householder reflections (dsytd2), one persistent cooperative kernel;
//   2. all m eigenvalues of T by bisection on Sturm counts (dstebz), one thread per index;
//   3. the top r eigenvectors of T by inverse iteration, re-orthogonalised within clusters (dstein), one CTA per cluster;
//   4. back-transformation x = Q z (dormtr), then the residual ||C x - lambda x|| against the fp32 C, sign, floor and fp32 outputs.
// No floating-point atomics: every reduction runs in a fixed order, so a given C gives the same bits on every call and every rank.
#include <algorithm>

#include "common.cuh"

namespace desmo {

constexpr int kTdThreads = 512;     // tridiagonalisation CTA: 16 warps, one row of the trailing matrix per warp at a time
constexpr int kEighThreads = 256;   // every other kernel
constexpr int kInvIters = 3;        // inverse-iteration solves per vector (dstein: converged + 2 extra)
constexpr double kEps = 0x1p-53;    // fp64 unit roundoff
constexpr size_t kEighHeadBytes = 256;  // head, padded

// workspace head (include/desmo_b200.h): {int32 status, int32 pad, double worst residual / lambda_1}, then the grid barrier counter
struct EighHead {
    int32_t status;
    int32_t pad;
    double residual;
    unsigned barrier;
};

__device__ __forceinline__ unsigned ld_acquire_gpu(const unsigned* p) {
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

// Grid-wide barrier of the cooperative tridiagonalisation kernel: a monotonic arrival counter (zeroed before the launch).  A CTA
// that never arrives fails the launch after ~10 s instead of hanging the GPU.
__device__ __forceinline__ void grid_barrier(unsigned* counter, unsigned& target) {
    __syncthreads();
    target += gridDim.x;
    if (threadIdx.x == 0) {
        __threadfence();
        atomicAdd(counter, 1u);
        const unsigned long long t0 = globaltimer_ns();
        while ((int)(ld_acquire_gpu(counter) - target) < 0)
            if (globaltimer_ns() - t0 > 10000000000ull) __trap();
        __threadfence();
    }
    __syncthreads();
}

// Fixed-order block sum (any blockDim.x that is a multiple of 32, at most 1024); every thread gets the result.
__device__ double eigh_block_sum(double v, double* sh) {
    v = warp_sum(v);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
    __syncthreads();
    double s = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += sh[w];
    __syncthreads();
    return s;
}
__device__ double eigh_block_max(double v, double* sh) {
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    __syncthreads();
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
    __syncthreads();
    double s = sh[0];
    for (int w = 1; w < (int)(blockDim.x >> 5); ++w) s = fmax(s, sh[w]);
    __syncthreads();
    return s;
}

// A[i][j] = C[max(i,j)][min(i,j)]: the lower triangle of the fp32 Gram, widened exactly (np.linalg.eigh's UPLO='L' reading)
__global__ void __launch_bounds__(kEighThreads) eigh_widen_kernel(int m, const float* __restrict__ C, double* __restrict__ A) {
    const long long e = (long long)blockIdx.x * kEighThreads + threadIdx.x;
    if (e >= (long long)m * m) return;
    const int i = (int)(e / m), j = (int)(e % m);
    A[e] = (double)(i >= j ? C[e] : C[(long long)j * m + i]);
}

// Householder tridiagonalisation (dsytd2, lower), A full symmetric storage, one persistent cooperative grid.
// Step k: H_k = I - tau_k v_k v_k^T with v_k[k+1] = 1 zeroes column k below the subdiagonal; p = tau A22 v, w = p - (tau/2)(p.v) v,
// A22 -= v w^T + w v^T.  The rank-2 update of step k - 1 is fused into the matrix-vector product of step k: one pass over the
// trailing matrix and one grid barrier per step.  Every CTA forms row k of the updated matrix, the reflector and w itself (in
// shared memory, fixed-order sums), so only p crosses CTAs.  v_k is kept in row k of A (columns k+1..m-1) for the back-transform.
// Data written by other CTAs is read with ld.global.cg (L2): rows change owner from step to step.
__global__ void __launch_bounds__(kTdThreads, 1) eigh_tridiag_kernel(int m, double* __restrict__ A, double* __restrict__ d,
                                                                      double* __restrict__ e, double* __restrict__ tau_out,
                                                                      double* __restrict__ pbuf, unsigned* __restrict__ counter) {
    extern __shared__ double sm[];
    __shared__ double red[32];
    double* vp = sm;          // v_{k-1} (zero outside k..m-1)
    double* wp = sm + m;      // w_{k-1}
    double* vc = sm + 2 * m;  // v_k
    const int tid = threadIdx.x, lane = tid & 31;
    const int gwarp = blockIdx.x * (kTdThreads / 32) + (tid >> 5), nwarps = gridDim.x * (kTdThreads / 32);
    for (int j = tid; j < m; j += kTdThreads) vp[j] = wp[j] = 0.0;
    __syncthreads();
    unsigned target = 0;
    for (int k = 0; k < m - 1; ++k) {
        // row k of A^(k) (the update of step k - 1 applied on the fly) -> d_k, the reflector of x = A^(k)[k+1:, k]
        const double vk = vp[k], wk = wp[k];
        double ss = 0.0;
        for (int j = k + tid; j < m; j += kTdThreads) {
            const double c = __ldcg(A + (size_t)k * m + j) - vk * wp[j] - wk * vp[j];
            vc[j] = c;
            if (j >= k + 2) ss += c * c;
        }
        ss = eigh_block_sum(ss, red);
        const double dk = vc[k], alpha = vc[k + 1];
        double beta = alpha, tau = 0.0, scale = 0.0;
        if (ss > 0.0) {
            beta = -copysign(sqrt(alpha * alpha + ss), alpha);
            tau = (beta - alpha) / beta;
            scale = 1.0 / (alpha - beta);
        }
        __syncthreads();
        for (int j = tid; j < m; j += kTdThreads) vc[j] = j <= k ? 0.0 : (j == k + 1 ? 1.0 : vc[j] * scale);
        if (blockIdx.x == 0) {
            if (tid == 0) { d[k] = dk; e[k] = beta; tau_out[k] = tau; }
            if (k > 0)  // row k - 1 was last read in step k - 1
                for (int j = k + tid; j < m; j += kTdThreads) A[(size_t)(k - 1) * m + j] = vp[j];
        }
        __syncthreads();
        // rows i > k: apply the update of step k - 1, store, and p_i = tau (A^(k) v_k)_i
        double* p = pbuf + (size_t)(k & 1) * m;
        for (int i = k + 1 + gwarp; i < m; i += nwarps) {
            const double vi = vp[i], wi = wp[i];
            double* Ai = A + (size_t)i * m;
            double acc = 0.0;
            for (int j = k + 1 + lane; j < m; j += 32) {
                const double x = __ldcg(Ai + j) - vi * wp[j] - wi * vp[j];
                Ai[j] = x;
                acc += x * vc[j];
            }
            acc = warp_sum(acc);
            if (lane == 0) p[i] = tau * acc;
        }
        grid_barrier(counter, target);
        // w_k = p - (tau / 2)(p . v_k) v_k, in every CTA
        double s = 0.0;
        for (int j = k + 1 + tid; j < m; j += kTdThreads) s += __ldcg(p + j) * vc[j];
        s = eigh_block_sum(s, red);
        const double h = 0.5 * tau * s;
        for (int j = tid; j < m; j += kTdThreads) wp[j] = j <= k ? 0.0 : __ldcg(p + j) - h * vc[j];
        double* t = vp; vp = vc; vc = t;
        __syncthreads();
    }
    if (blockIdx.x == 0 && tid == 0) {
        d[m - 1] = __ldcg(A + (size_t)(m - 1) * m + m - 1) - 2.0 * vp[m - 1] * wp[m - 1];
        if (m >= 2) A[(size_t)(m - 2) * m + m - 1] = 1.0;  // v_{m-2} (tau = 0)
    }
}

// Number of eigenvalues of T below x (dlaebz's Sturm count with the pivmin guard).  e2[i] = e_i^2.
__device__ __forceinline__ int sturm_count(int m, const double* __restrict__ d, const double* __restrict__ e2, double x, double pivmin) {
    double q = d[0] - x;
    if (fabs(q) < pivmin) q = -pivmin;
    int c = q <= 0.0;
    for (int i = 1; i < m; ++i) {
        q = (d[i] - x) - e2[i - 1] / q;
        if (fabs(q) < pivmin) q = -pivmin;
        c += q <= 0.0;
    }
    return c;
}

struct TriNorm { double gl, gu, tnorm, pivmin; };

__device__ TriNorm tri_bounds(int m, const double* __restrict__ d, const double* __restrict__ e) {
    double gl = d[0], gu = d[0], emax2 = 0.0;
    for (int i = 0; i < m; ++i) {
        const double el = i > 0 ? fabs(e[i - 1]) : 0.0, er = i < m - 1 ? fabs(e[i]) : 0.0;
        gl = fmin(gl, d[i] - el - er);
        gu = fmax(gu, d[i] + el + er);
        emax2 = fmax(emax2, er * er);
    }
    TriNorm t;
    t.tnorm = fmax(fabs(gl), fabs(gu));
    t.pivmin = 0x1p-1022 * fmax(1.0, emax2);
    t.gl = gl - 2.1 * t.tnorm * kEps * m - 4.2 * t.pivmin;
    t.gu = gu + 2.1 * t.tnorm * kEps * m + 4.2 * t.pivmin;
    return t;
}

__global__ void __launch_bounds__(kEighThreads) eigh_e2_kernel(int m, const double* __restrict__ e, double* __restrict__ e2) {
    const int i = blockIdx.x * kEighThreads + threadIdx.x;
    if (i < m - 1) e2[i] = e[i] * e[i];
}

// eigenvalue i (ascending) of T by bisection, to max(eps ||T||, 2 eps |lambda|) (dstebz with abstol = eps ||T||_1)
__global__ void __launch_bounds__(kEighThreads) eigh_bisect_kernel(int m, const double* __restrict__ d, const double* __restrict__ e,
                                                                   const double* __restrict__ e2, double* __restrict__ lam) {
    const int i = blockIdx.x * kEighThreads + threadIdx.x;
    if (i >= m) return;
    const TriNorm t = tri_bounds(m, d, e);
    const double atol = fmax(kEps * t.tnorm, t.pivmin);
    double lo = t.gl, hi = t.gu;
    for (int it = 0; it < 256; ++it) {
        if (hi - lo <= fmax(atol, 2.0 * kEps * fmax(fabs(lo), fabs(hi)))) break;
        const double mid = 0.5 * (lo + hi);
        if (mid <= lo || mid >= hi) break;
        if (sturm_count(m, d, e2, mid, t.pivmin) > i) hi = mid; else lo = mid;
    }
    lam[i] = 0.5 * (lo + hi);
}

// The bisection intervals of neighbouring indices may overlap by the tolerance: sort (insertion sort: O(m) on sorted input).
__global__ void eigh_sort_kernel(int m, double* __restrict__ lam) {
    for (int i = 1; i < m; ++i) {
        const double x = lam[i];
        int j = i - 1;
        while (j >= 0 && lam[j] > x) { lam[j + 1] = lam[j]; --j; }
        lam[j + 1] = x;
    }
}

__device__ __forceinline__ double start_entry(int q, int t) {  // deterministic start vector in (-1, 1)
    unsigned h = (unsigned)(t * 2654435761u) ^ (unsigned)((q + 1) * 40503u) ^ 0x9e3779b9u;
    h ^= h >> 13; h *= 0x5bd1e995u; h ^= h >> 15;
    return (double)(h & 0xffffff) / 8388608.0 - 1.0;
}

// Inverse iteration for the top r eigenvalues (descending index q = 0..r-1 is lam[m-1-q]), one CTA per cluster (dstein): a new
// cluster starts where neighbours differ by more than 1e-3 ||T||_1; shifts closer than 10 eps |lambda| are pulled apart.  Each
// vector: LU with partial pivoting of T - x I (thread 0; tiny pivots raised to eps ||T||), kInvIters solves from a seeded start,
// each followed by re-orthogonalisation against the cluster's earlier vectors (CGS2) and a normalisation.  LU factors in `lu` [r][5][m].
__global__ void __launch_bounds__(kEighThreads) eigh_inviter_kernel(int m, int r, const double* __restrict__ d,
                                                                    const double* __restrict__ e, const double* __restrict__ lam,
                                                                    double* __restrict__ Z, double* __restrict__ lu) {
    extern __shared__ double b[];  // [m]
    __shared__ double red[32];
    __shared__ int range[2];
    __shared__ double proj[DESMO_MAX_R];
    const int tid = threadIdx.x;
    double onenrm = 0.0;
    for (int i = tid; i < m; i += kEighThreads)
        onenrm = fmax(onenrm, fabs(d[i]) + (i > 0 ? fabs(e[i - 1]) : 0.0) + (i < m - 1 ? fabs(e[i]) : 0.0));
    onenrm = eigh_block_max(onenrm, red);
    const double ortol = 1e-3 * onenrm, ptiny = fmax(kEps * onenrm, 0x1p-1000);
    if (tid == 0) {
        int c = -1, q0 = -1, q1 = -1;
        for (int q = 0; q < r; ++q) {
            if (q == 0 || lam[m - q] - lam[m - 1 - q] > ortol) {
                if (++c == (int)blockIdx.x) q0 = q; else if (c == (int)blockIdx.x + 1) { q1 = q; break; }
            }
        }
        range[0] = q0;
        range[1] = (q0 >= 0 && q1 < 0) ? r : q1;
    }
    __syncthreads();
    const int q0 = range[0], q1 = range[1];
    if (q0 < 0) return;
    double* u0 = lu + (size_t)blockIdx.x * 5 * m;  // 1 / pivot: the solves multiply (no division on their dependency chain)
    double* u1 = u0 + m;
    double* u2 = u1 + m;
    double* l = u2 + m;
    double* sw = l + m;  // 1.0 where rows i and i + 1 were swapped
    double xprev = 0.0;
    for (int q = q0; q < q1; ++q) {
        double x = lam[m - 1 - q];
        if (q > q0 && xprev - x < 10.0 * kEps * fabs(x)) x = xprev - 10.0 * kEps * fabs(x);
        xprev = x;
        if (tid == 0) {
            double x0 = d[0] - x, x1 = m > 1 ? e[0] : 0.0;  // current row: x0 at column i, x1 at column i + 1
            for (int i = 0; i < m - 1; ++i) {
                const double ei = e[i], ai = d[i + 1] - x, en = i + 1 < m - 1 ? e[i + 1] : 0.0;
                if (fabs(x0) >= fabs(ei)) {
                    const double piv = fabs(x0) < ptiny ? copysign(ptiny, x0) : x0;
                    const double li = ei / piv;
                    u0[i] = 1.0 / piv; u1[i] = x1; u2[i] = 0.0; l[i] = li; sw[i] = 0.0;
                    x0 = ai - li * x1; x1 = en;
                } else {
                    const double li = x0 / ei;
                    u0[i] = 1.0 / ei; u1[i] = ai; u2[i] = en; l[i] = li; sw[i] = 1.0;
                    x0 = x1 - li * ai; x1 = -li * en;
                }
            }
            u0[m - 1] = 1.0 / (fabs(x0) < ptiny ? copysign(ptiny, x0) : x0);
        }
        for (int t = tid; t < m; t += kEighThreads) b[t] = start_entry(q, t);
        __syncthreads();
        for (int it = 0; it < kInvIters; ++it) {
            if (tid == 0) {
                for (int i = 0; i < m - 1; ++i) {
                    if (sw[i] != 0.0) { const double t = b[i]; b[i] = b[i + 1]; b[i + 1] = t - l[i] * b[i]; }
                    else b[i + 1] -= l[i] * b[i];
                }
                b[m - 1] *= u0[m - 1];
                if (m > 1) b[m - 2] = (b[m - 2] - u1[m - 2] * b[m - 1]) * u0[m - 2];
                for (int i = m - 3; i >= 0; --i) b[i] = (b[i] - u1[i] * b[i + 1] - u2[i] * b[i + 2]) * u0[i];
            }
            __syncthreads();
            // two classical Gram-Schmidt passes: all projections of a pass in one sweep (one warp per earlier vector, lanes in a fixed
            // order), so a vector costs two barriers per pass instead of one block reduction per earlier vector
            for (int pass = 0; pass < 2 && q > q0; ++pass) {
                for (int p = q0 + (tid >> 5); p < q; p += kEighThreads / 32) {
                    const double* zp = Z + (size_t)p * m;
                    double s = 0.0;
                    for (int t = tid & 31; t < m; t += 32) s += zp[t] * b[t];
                    s = warp_sum(s);
                    if ((tid & 31) == 0) proj[p - q0] = s;
                }
                __syncthreads();
                for (int t = tid; t < m; t += kEighThreads) {
                    double v = b[t];
                    for (int p = q0; p < q; ++p) v -= proj[p - q0] * Z[(size_t)p * m + t];
                    b[t] = v;
                }
                __syncthreads();
            }
            double nn = 0.0;
            for (int t = tid; t < m; t += kEighThreads) nn += b[t] * b[t];
            nn = eigh_block_sum(nn, red);
            const double inv = nn > 0.0 ? 1.0 / sqrt(nn) : 0.0;
            for (int t = tid; t < m; t += kEighThreads) b[t] *= inv;
            __syncthreads();
        }
        for (int t = tid; t < m; t += kEighThreads) Z[(size_t)q * m + t] = b[t];
        __syncthreads();
    }
}

// x = H_0 H_1 ... H_{m-2} z for each of the r vectors (one CTA each); v_k is row k of A from column k + 1 on.
__global__ void __launch_bounds__(kEighThreads) eigh_backtransform_kernel(int m, const double* __restrict__ A,
                                                                          const double* __restrict__ tau, double* __restrict__ Z) {
    extern __shared__ double z[];  // [m]
    __shared__ double red[32];
    double* zg = Z + (size_t)blockIdx.x * m;
    for (int t = threadIdx.x; t < m; t += kEighThreads) z[t] = zg[t];
    __syncthreads();
    for (int k = m - 2; k >= 0; --k) {
        const double tk = tau[k];
        if (tk == 0.0) continue;
        const double* v = A + (size_t)k * m;
        double s = 0.0;
        for (int t = k + 1 + threadIdx.x; t < m; t += kEighThreads) s += v[t] * z[t];
        s = tk * eigh_block_sum(s, red);
        for (int t = k + 1 + threadIdx.x; t < m; t += kEighThreads) z[t] -= s * v[t];
        __syncthreads();
    }
    for (int t = threadIdx.x; t < m; t += kEighThreads) zg[t] = z[t];
}

// Y[q][t] = sum_s C[t][s] X[q][s] in fp64 over the fp32 C read as in eigh_widen_kernel: 32 rows x 16 vectors per CTA, C through a
// 32 x 32 shared tile loaded along whichever of C[t][s] / C[s][t] is the lower triangle (coalesced either way).
constexpr int kMvRows = 32, kMvVecs = 16;
__global__ void __launch_bounds__(kEighThreads) eigh_matvec_kernel(int m, int r, const float* __restrict__ C, const double* __restrict__ X,
                                                                   double* __restrict__ Y) {
    __shared__ float Ct[kMvRows][kMvRows + 1];
    __shared__ double Xs[kMvVecs][kMvRows];
    const int t0 = blockIdx.x * kMvRows, q0 = blockIdx.y * kMvVecs;
    const int tid = threadIdx.x, ty = tid >> 5, tx = tid & 31;  // 8 x 32
    double acc[2] = {0.0, 0.0};  // row t0 + tx, vectors q0 + ty and q0 + ty + 8
    for (int s0 = 0; s0 < m; s0 += kMvRows) {
        for (int a = ty; a < kMvRows; a += 8) {
            // lower-triangle tile (t >= s): C[t][s] with s along the lanes; upper: C[s][t] with t along the lanes
            if (t0 >= s0) {
                const int t = t0 + a, s = s0 + tx;
                Ct[a][tx] = (t < m && s < m) ? (t >= s ? C[(size_t)t * m + s] : C[(size_t)s * m + t]) : 0.0f;
            } else {
                const int s = s0 + a, t = t0 + tx;
                Ct[tx][a] = (t < m && s < m) ? C[(size_t)s * m + t] : 0.0f;
            }
        }
        for (int a = ty; a < kMvVecs; a += 8) {
            const int q = q0 + a, s = s0 + tx;
            Xs[a][tx] = (q < r && s < m) ? X[(size_t)q * m + s] : 0.0;
        }
        __syncthreads();
#pragma unroll 8
        for (int s = 0; s < kMvRows; ++s) {
            const double c = (double)Ct[tx][s];
            acc[0] += c * Xs[ty][s];
            acc[1] += c * Xs[ty + 8][s];
        }
        __syncthreads();
    }
    const int t = t0 + tx;
    if (t < m) {
        if (q0 + ty < r) Y[(size_t)(q0 + ty) * m + t] = acc[0];
        if (q0 + ty + 8 < r) Y[(size_t)(q0 + ty + 8) * m + t] = acc[1];
    }
}

// per vector q: residual ||y - lambda x||, sign (largest-|.| entry positive; ties to the positive entry, as eig_ritz_kernel), fp32 row
__global__ void __launch_bounds__(kEighThreads) eigh_emit_kernel(int m, const double* __restrict__ lam, const double* __restrict__ X,
                                                                 const double* __restrict__ Y, float* __restrict__ V, double* __restrict__ res) {
    __shared__ double red[32];
    const int q = blockIdx.x;
    const double* x = X + (size_t)q * m;
    const double* y = Y + (size_t)q * m;
    const double th = lam[m - 1 - q];
    double r2 = 0.0, best = 0.0;
    for (int t = threadIdx.x; t < m; t += kEighThreads) {
        const double v = x[t], dv = y[t] - th * v;
        r2 += dv * dv;
        if (fabs(v) > fabs(best)) best = v;
    }
    r2 = eigh_block_sum(r2, red);
    double cand = best;
    for (int o = 16; o > 0; o >>= 1) {
        const double other = __shfl_xor_sync(0xffffffffu, cand, o);
        if (fabs(other) > fabs(cand) || (fabs(other) == fabs(cand) && other > cand)) cand = other;
    }
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = cand;
    __syncthreads();
    double top = red[0];
    for (int w = 1; w < kEighThreads / 32; ++w)
        if (fabs(red[w]) > fabs(top) || (fabs(red[w]) == fabs(top) && red[w] > top)) top = red[w];
    const double flip = top < 0.0 ? -1.0 : 1.0;
    for (int t = threadIdx.x; t < m; t += kEighThreads) V[(size_t)q * m + t] = (float)(flip * x[t]);
    if (threadIdx.x == 0) res[q] = sqrt(r2);
}

// S (all m, descending, floored), sigma = fp32 S[:r], and the report: worst residual / lambda_1 over the live modes, status
__global__ void __launch_bounds__(1024) eigh_finish_kernel(int m, int r, const float* __restrict__ C, const double* __restrict__ lam,
                                                           const double* __restrict__ res, double* __restrict__ S, float* __restrict__ sigma,
                                                           EighHead* __restrict__ head) {
    __shared__ double red[32];
    double tr = 0.0;
    for (int t = threadIdx.x; t < m; t += 1024) tr += (double)C[(size_t)t * m + t];
    tr = eigh_block_sum(tr, red);
    const double floor_lam = 0x1p-23 * tr, lam1 = lam[m - 1];
    for (int i = threadIdx.x; i < m; i += 1024) {
        const double li = lam[m - 1 - i];
        const double s = li > floor_lam ? sqrt(li) : 0.0;
        S[i] = s;
        if (i < r) sigma[i] = (float)s;
    }
    if (threadIdx.x == 0) {
        double worst = 0.0;
        bool finite = isfinite(tr) && isfinite(lam1);
        for (int q = 0; q < r; ++q) {
            finite = finite && isfinite(res[q]);
            if (lam[m - 1 - q] > floor_lam) worst = fmax(worst, res[q] / lam1);
        }
        head->status = finite ? 0 : 1;
        head->residual = finite ? worst : __longlong_as_double(0x7ff8000000000000ll);
    }
}

struct EighLayout {
    EighHead* head;
    double *A, *d, *e, *e2, *tau, *p, *lam, *Z, *Y, *res, *lu;
};

static EighLayout eigh_layout(int m, int r, void* ws) {
    EighLayout L;
    L.head = static_cast<EighHead*>(ws);
    double* q = reinterpret_cast<double*>(static_cast<char*>(ws) + kEighHeadBytes);
    L.A = q; q += (size_t)m * m;
    L.d = q; q += m;
    L.e = q; q += m;
    L.e2 = q; q += m;
    L.tau = q; q += m;
    L.p = q; q += 2 * (size_t)m;
    L.lam = q; q += m;
    L.Z = q; q += (size_t)r * m;
    L.Y = q; q += (size_t)r * m;
    L.res = q; q += r;
    L.lu = q;
    return L;
}

size_t pod_eigh_workspace_bytes(int m, int r) {
    return kEighHeadBytes + sizeof(double) * ((size_t)m * m + 7 * (size_t)m + (size_t)r * (7 * (size_t)m + 1));
}

int pod_eigh(int m, int r, const float* C, double* S, float* V, float* sigma, void* workspace, cudaStream_t st) {
    const EighLayout L = eigh_layout(m, r, workspace);
    DESMO_CUDA(cudaMemsetAsync(workspace, 0, kEighHeadBytes, st));
    const long long mm = (long long)m * m;
    eigh_widen_kernel<<<(unsigned)((mm + kEighThreads - 1) / kEighThreads), kEighThreads, 0, st>>>(m, C, L.A);
    DESMO_CUDA(cudaGetLastError());

    // tridiagonalisation: as many CTAs as fit (one per SM), at most one warp per row of the first step
    const size_t smem = 3 * sizeof(double) * (size_t)m;
    DESMO_CUDA(cudaFuncSetAttribute(eigh_tridiag_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int dev = 0, sms = 0, per_sm = 0;
    DESMO_CUDA(cudaGetDevice(&dev));
    DESMO_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    DESMO_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, eigh_tridiag_kernel, kTdThreads, smem));
    if (per_sm < 1) { set_error("pod_eigh: the tridiagonalisation kernel does not fit an SM at m=%d", m); return DESMO_ERR_CUDA; }
    const int grid = std::max(1, std::min(sms, (m + kTdThreads / 32 - 1) / (kTdThreads / 32)));
    {
        int mm_ = m;
        unsigned* counter = &L.head->barrier;
        double *A = L.A, *d = L.d, *e = L.e, *tau = L.tau, *p = L.p;
        void* args[] = {&mm_, &A, &d, &e, &tau, &p, &counter};
        DESMO_CUDA(cudaLaunchCooperativeKernel((const void*)eigh_tridiag_kernel, dim3(grid), dim3(kTdThreads), args, smem, st));
    }
    eigh_e2_kernel<<<(m + kEighThreads - 1) / kEighThreads, kEighThreads, 0, st>>>(m, L.e, L.e2);
    eigh_bisect_kernel<<<(m + kEighThreads - 1) / kEighThreads, kEighThreads, 0, st>>>(m, L.d, L.e, L.e2, L.lam);
    eigh_sort_kernel<<<1, 1, 0, st>>>(m, L.lam);
    DESMO_CUDA(cudaGetLastError());

    const size_t vsmem = sizeof(double) * (size_t)m;
    DESMO_CUDA(cudaFuncSetAttribute(eigh_inviter_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)vsmem));
    DESMO_CUDA(cudaFuncSetAttribute(eigh_backtransform_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)vsmem));
    eigh_inviter_kernel<<<r, kEighThreads, vsmem, st>>>(m, r, L.d, L.e, L.lam, L.Z, L.lu);
    eigh_backtransform_kernel<<<r, kEighThreads, vsmem, st>>>(m, L.A, L.tau, L.Z);
    eigh_matvec_kernel<<<dim3((m + kMvRows - 1) / kMvRows, (r + kMvVecs - 1) / kMvVecs), kEighThreads, 0, st>>>(m, r, C, L.Z, L.Y);
    eigh_emit_kernel<<<r, kEighThreads, 0, st>>>(m, L.lam, L.Z, L.Y, V, L.res);
    eigh_finish_kernel<<<1, 1024, 0, st>>>(m, r, C, L.lam, L.res, S, sigma, L.head);
    DESMO_CUDA(cudaGetLastError());
    return DESMO_OK;
}

}  // namespace desmo
