// POD initialisation by the method of snapshots (replaces np.linalg.svd of the n x m data matrix, CYL:197-205):
//   C = U U^T (m x m Gram over mesh points; the one dense contraction)  ->  top-r eigenpairs (lambda_i, v_i) on device
//   ->  POD mode i = X v_i / sqrt(lambda_i), i.e. P[i][x] = sum_t U[t][x] v_i[t] / sigma_i.
// Point-sharded: each rank forms the Gram of its slab, one all-reduce of C, replicated eigensolve, local projection.
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
// Top-r eigenpairs of the (all-reduced) Gram: block subspace iteration with b = r + 8 vectors in fp64,
// modified Gram-Schmidt each sweep, Rayleigh-Ritz (cyclic Jacobi on the b x b projection) at the end.
// ---------------------------------------------------------------------------------------------------------------
constexpr int kEigMaxB = 16;

__global__ void __launch_bounds__(256) eig_init_kernel(int m, int b, double* V) {
    // deterministic, well-spread start: V[j][t] = cos(pi (j+1)(t+0.5)/m) + small hash noise
    const int t = blockIdx.x * 256 + threadIdx.x;
    if (t >= m) return;
    for (int j = 0; j < b; ++j) {
        unsigned h = (unsigned)(t * 2654435761u) ^ (unsigned)((j + 1) * 40503u);
        h ^= h >> 13; h *= 0x5bd1e995u; h ^= h >> 15;
        V[(size_t)j * m + t] = cos(3.141592653589793 * (j + 1) * (t + 0.5) / m) + 1e-3 * ((double)(h & 0xffff) / 65536.0 - 0.5);
    }
}

// Y[j][t] = sum_s C[t][s] V[j][s]   (one warp per row t)
__global__ void __launch_bounds__(256) eig_matvec_kernel(int m, int b, const float* __restrict__ C, const double* __restrict__ V,
                                                         double* __restrict__ Y) {
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
__global__ void __launch_bounds__(1024) eig_orth_kernel(int m, int b, const double* __restrict__ Y, double* __restrict__ V) {
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

// Rayleigh-Ritz: H = V^T (C V) = V^T Y (b x b), Jacobi eigen-decomposition, rotate, sort, sign-normalise, emit top r.
__global__ void __launch_bounds__(1024) eig_ritz_kernel(int m, int b, int r, const double* __restrict__ V, const double* __restrict__ Y,
                                                        float* __restrict__ Vout, float* __restrict__ sigma) {
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
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int i = 0; i < b; ++i)
            for (int j = 0; j < b; ++j) Q[i][j] = (i == j) ? 1.0 : 0.0;
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
                    for (int k = 0; k < b; ++k) {
                        const double hkp = H[k][p], hkq = H[k][q];
                        H[k][p] = c * hkp - s2 * hkq;
                        H[k][q] = s2 * hkp + c * hkq;
                    }
                    for (int k = 0; k < b; ++k) {
                        const double hpk = H[p][k], hqk = H[q][k];
                        H[p][k] = c * hpk - s2 * hqk;
                        H[q][k] = s2 * hpk + c * hqk;
                    }
                    for (int k = 0; k < b; ++k) {
                        const double qkp = Q[k][p], qkq = Q[k][q];
                        Q[k][p] = c * qkp - s2 * qkq;
                        Q[k][q] = s2 * qkp + c * qkq;
                    }
                }
        }
        for (int i = 0; i < b; ++i) order[i] = i;
        for (int i = 0; i < b; ++i)
            for (int j = i + 1; j < b; ++j)
                if (H[order[j]][order[j]] > H[order[i]][order[i]]) { const int tmp = order[i]; order[i] = order[j]; order[j] = tmp; }
    }
    __syncthreads();
    for (int i = 0; i < r; ++i) {
        const int col = order[i];
        // ritz vector = sum_j Q[j][col] V[j]; find the largest-|.| entry for the sign convention
        double best = 0.0;
        for (int t = threadIdx.x; t < m; t += 1024) {
            double v = 0.0;
            for (int j = 0; j < b; ++j) v += Q[j][col] * V[(size_t)j * m + t];
            if (fabs(v) > fabs(best)) best = v;
        }
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
        if (threadIdx.x == 0) sigma[i] = (float)sqrt(fmax(H[col][col], 0.0));
        __syncthreads();
    }
}

int pod_eig(int m, int r, const float* C, float* V, float* sigma, void* workspace, size_t workspace_bytes, cudaStream_t st) {
    const int b = (r + 8 <= kEigMaxB) ? r + 8 : kEigMaxB;
    if (r > kEigMaxB - 2 || b > m) { set_error("pod_eig: r=%d unsupported for m=%d", r, m); return DESMO_ERR_UNSUPPORTED; }
    const size_t need = 2 * sizeof(double) * (size_t)b * m;
    if (workspace_bytes < need) { set_error("pod_eig: workspace too small (%zu < %zu)", workspace_bytes, need); return DESMO_ERR_ARG; }
    double* Vd = static_cast<double*>(workspace);
    double* Yd = Vd + (size_t)b * m;
    eig_init_kernel<<<(m + 255) / 256, 256, 0, st>>>(m, b, Yd);
    eig_orth_kernel<<<1, 1024, 0, st>>>(m, b, Yd, Vd);
    const int iters = 120;
    for (int it = 0; it < iters; ++it) {
        eig_matvec_kernel<<<(m + 7) / 8, 256, 0, st>>>(m, b, C, Vd, Yd);
        eig_orth_kernel<<<1, 1024, 0, st>>>(m, b, Yd, Vd);
    }
    eig_matvec_kernel<<<(m + 7) / 8, 256, 0, st>>>(m, b, C, Vd, Yd);
    eig_ritz_kernel<<<1, 1024, 0, st>>>(m, b, r, Vd, Yd, V, sigma);
    DESMO_CUDA(cudaGetLastError());
    return DESMO_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// Back-projection: P[i][x] = sum_t U[t][x] V[i][t] / sigma_i   (streams U once, HBM-bound)
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
    extern __shared__ float Vs[];  // [m][kMaxR]
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
                const float inv = 1.0f / sigma[i];
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
    pod_project_kernel<UT><<<(unsigned)g, 256, smem, st>>>(U, s->ld, s->n, s->m, s->r, V, sigma, P);
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
