// Snapshot pre-processing on the device (SURVEY.md section 8f-2): what the reference does in numpy between the VTK reader and
// the POD / training loop --
//   convert3Dto2D_data (CYL:88-106)  : drop the w component of a 2-D flow          -> d_use = 2 of d_in = 3
//   convertToMagnitude (CYL:109-133) : |u| per point and snapshot, in float64       -> DESMO_PRE_MAGNITUDE
//   subtract_mean      (CYL:136-149) : remove the temporal mean of every point      -> DESMO_PRE_SUBTRACT_MEAN
//   ... * 1/sqrt(m)    (ANEU:143)    : the aneurysm scripts' extra scaling          -> DESMO_PRE_SCALE_SQRT_M
//   X[:, 0::2]         (TURB:189)    : keep every t_stride-th snapshot AFTER the mean was taken over all of them
//   X.T -> FloatTensor (CYL:356,708) : time-major fp32 snapshot, here straight into the padded U[m][ld] layout
// The raw input is X.T as the reader produces it: V[m_in][n * d_in], the components of a point adjacent.  One thread owns one
// point; pass 1 accumulates the fp64 temporal sum, pass 2 recomputes the magnitude and rounds (|u| - mean) * scale to fp32 ONCE,
// exactly where the reference's float64 -> float32 cast sits.  HBM-bound: (2 * d_in * m_in * sizeof(in) + 4 * m) bytes / point.
// bf16 storage rounds that fp32 value once more (round to nearest even), i.e. it stores what fp32 preprocessing followed by torch's
// .bfloat16() stores.  snapshot_to_bf16 below is the same conversion for snapshots that are already fp32.
//
// Quantisation sums (optional, fp64 [2] += {sum (u - q)^2, sum u^2} over the real points, u the fp32 value, q the bf16 one): every
// block reduces its threads' sums in a fixed order into a partial of its own, and one block adds the partials in a fixed order, so
// the reported error is the same from run to run.
#include "common.cuh"

namespace desmo {

template <typename TIn>
__device__ __forceinline__ double point_value(const TIn* __restrict__ p, int d_use, bool magnitude) {
    if (!magnitude) return (double)p[0];
    // np.sum(np.square(Ui), 1) then np.sqrt, float64, no contraction into FMAs
    double s = __dmul_rn((double)p[0], (double)p[0]);
    for (int c = 1; c < d_use; ++c) s = __dadd_rn(s, __dmul_rn((double)p[c], (double)p[c]));
    return sqrt(s);
}

// sums of the 256 threads of a block, reduced in a fixed order; every thread of the block must call it
__device__ __forceinline__ void block_qsums(double e2, double u2, double* __restrict__ out) {
    __shared__ double sm[2][256];
    sm[0][threadIdx.x] = e2;
    sm[1][threadIdx.x] = u2;
    __syncthreads();
    for (int w = 128; w > 0; w >>= 1) {
        if ((int)threadIdx.x < w) {
            sm[0][threadIdx.x] += sm[0][threadIdx.x + w];
            sm[1][threadIdx.x] += sm[1][threadIdx.x + w];
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        out[0] = sm[0][0];
        out[1] = sm[1][0];
    }
}

__device__ __forceinline__ double* block_part(double* part) {
    return part + 2 * ((long long)blockIdx.y * gridDim.x + blockIdx.x);
}

// qsums += the sum of the nparts block partials (one block, fixed order)
__global__ void __launch_bounds__(256) qsums_finish_kernel(const double* __restrict__ part, long long nparts, double* __restrict__ qsums) {
    double e2 = 0.0, u2 = 0.0;
    for (long long i = threadIdx.x; i < nparts; i += 256) {
        e2 += part[2 * i];
        u2 += part[2 * i + 1];
    }
    __shared__ double tot[2];
    block_qsums(e2, u2, tot);
    if (threadIdx.x == 0) {
        qsums[0] += tot[0];
        qsums[1] += tot[1];
    }
}

// temporal mean of one point over all m_in input snapshots (0 without DESMO_PRE_SUBTRACT_MEAN)
template <typename TIn>
__device__ __forceinline__ double point_mean(const TIn* __restrict__ col, long long v_ld, int m_in, int d_use, int flags, bool magnitude) {
    double mean = 0.0;
    if (flags & DESMO_PRE_SUBTRACT_MEAN) {
        double acc[4] = {0.0, 0.0, 0.0, 0.0};
        int t = 0;
        for (; t + 4 <= m_in; t += 4) {
#pragma unroll
            for (int u = 0; u < 4; ++u) acc[u] += point_value(col + (long long)(t + u) * v_ld, d_use, magnitude);
        }
        for (; t < m_in; ++t) acc[0] += point_value(col + (long long)t * v_ld, d_use, magnitude);
        mean = ((acc[0] + acc[1]) + (acc[2] + acc[3])) / (double)m_in;
    }
    return mean;
}

template <typename TIn>
__global__ void __launch_bounds__(256) preprocess_kernel(const TIn* __restrict__ V, long long v_ld, long long n, long long ld, int m_in,
                                                         int m_out, int t_stride, int d_in, int d_use, int flags,
                                                         float* __restrict__ U, double* __restrict__ mean_out) {
    const long long x = (long long)blockIdx.x * 256 + threadIdx.x;
    if (x >= ld) return;
    if (x >= n) {
        for (int t = 0; t < m_out; ++t) U[(long long)t * ld + x] = 0.0f;
        return;
    }
    const bool magnitude = flags & DESMO_PRE_MAGNITUDE;
    const TIn* col = V + x * d_in;
    const double mean = point_mean(col, v_ld, m_in, d_use, flags, magnitude);
    if (mean_out) mean_out[x] = mean;
    const double scale = (flags & DESMO_PRE_SCALE_SQRT_M) ? 1.0 / sqrt((double)m_in) : 1.0;
#pragma unroll 4
    for (int t = 0; t < m_out; ++t) {
        const double v = point_value(col + (long long)t * t_stride * v_ld, d_use, magnitude);
        U[(long long)t * ld + x] = (float)(scale * (v - mean));  // (1/np.sqrt(m)) * (X - mean), one rounding to fp32
    }
}

// the same with bf16 output: the fp32 value above, rounded to nearest even once more; quantisation sums into qpart (may be NULL)
template <typename TIn>
__global__ void __launch_bounds__(256) preprocess_bf16_kernel(const TIn* __restrict__ V, long long v_ld, long long n, long long ld, int m_in,
                                                              int m_out, int t_stride, int d_in, int d_use, int flags,
                                                              __nv_bfloat16* __restrict__ U, double* __restrict__ mean_out,
                                                              double* __restrict__ qpart) {
    const long long x = (long long)blockIdx.x * 256 + threadIdx.x;
    double e2 = 0.0, u2 = 0.0;
    if (x >= n) {
        if (x < ld)
            for (int t = 0; t < m_out; ++t) U[(long long)t * ld + x] = __float2bfloat16_rn(0.0f);
    } else {
        const bool magnitude = flags & DESMO_PRE_MAGNITUDE;
        const TIn* col = V + x * d_in;
        const double mean = point_mean(col, v_ld, m_in, d_use, flags, magnitude);
        if (mean_out) mean_out[x] = mean;
        const double scale = (flags & DESMO_PRE_SCALE_SQRT_M) ? 1.0 / sqrt((double)m_in) : 1.0;
#pragma unroll 4
        for (int t = 0; t < m_out; ++t) {
            const double v = point_value(col + (long long)t * t_stride * v_ld, d_use, magnitude);
            const float u = (float)(scale * (v - mean));
            const __nv_bfloat16 q = __float2bfloat16_rn(u);
            U[(long long)t * ld + x] = q;
            const double d = (double)u - (double)__bfloat162float(q);
            e2 = fma(d, d, e2);
            u2 = fma((double)u, (double)u, u2);
        }
    }
    if (qpart) block_qsums(e2, u2, block_part(qpart));
}

// thread <-> two adjacent points (x, x + 1) of row t0 + y: one cvt.rn.bf16x2.f32 and one 4-byte store per row
__global__ void __launch_bounds__(256) snapshot_to_bf16_kernel(const float* __restrict__ src, long long src_ld, long long n, long long ld,
                                                               int t0, int rows, __nv_bfloat16* __restrict__ U, double* __restrict__ qpart) {
    const long long x = 2 * ((long long)blockIdx.x * 256 + threadIdx.x);
    double e2 = 0.0, u2 = 0.0;
    if (x < ld) {
        for (int y = blockIdx.y; y < rows; y += gridDim.y) {
            const float* row = src + (long long)y * src_ld;
            const float u0 = x < n ? row[x] : 0.0f, u1 = x + 1 < n ? row[x + 1] : 0.0f;
            uint32_t w;
            asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(w) : "f"(u1), "f"(u0));
            *reinterpret_cast<uint32_t*>(U + (long long)(t0 + y) * ld + x) = w;
            const double d0 = (double)u0 - (double)__uint_as_float(w << 16), d1 = (double)u1 - (double)__uint_as_float(w & 0xffff0000u);
            e2 = fma(d1, d1, fma(d0, d0, e2));
            u2 = fma((double)u1, (double)u1, fma((double)u0, (double)u0, u2));
        }
    }
    if (qpart) block_qsums(e2, u2, block_part(qpart));
}

// per-block partials of the quantisation sums live in stream-ordered scratch (the entry points take no workspace)
static int qsums_begin(double* qsums, long long nblocks, double** part, cudaStream_t st) {
    *part = nullptr;
    if (qsums) DESMO_CUDA(cudaMallocAsync(reinterpret_cast<void**>(part), sizeof(double) * 2 * (size_t)nblocks, st));
    return DESMO_OK;
}
static int qsums_end(double* qsums, long long nblocks, double* part, cudaStream_t st) {
    if (!qsums) return DESMO_OK;
    qsums_finish_kernel<<<1, 256, 0, st>>>(part, nblocks, qsums);
    DESMO_CUDA(cudaGetLastError());
    DESMO_CUDA(cudaFreeAsync(part, st));
    return DESMO_OK;
}

int snapshot_to_bf16(const desmo_shape* s, const float* src, long long src_ld, int t0, int rows, __nv_bfloat16* U, double* qsums,
                     cudaStream_t st) {
    const dim3 grid((unsigned)((s->ld / 2 + 255) / 256), (unsigned)(rows < 64 ? rows : 64));
    const long long nb = (long long)grid.x * grid.y;
    double* part;
    int rc = qsums_begin(qsums, nb, &part, st);
    if (rc) return rc;
    snapshot_to_bf16_kernel<<<grid, 256, 0, st>>>(src, src_ld, s->n, s->ld, t0, rows, U, part);
    DESMO_CUDA(cudaGetLastError());
    return qsums_end(qsums, nb, part, st);
}

int preprocess(const desmo_shape* s, const void* V, int v_dtype, long long v_ld, int m_in, int t_stride, int d_in, int d_use, int flags,
               void* U, int u_dtype, double* qsums, double* mean, cudaStream_t st) {
    const unsigned grid = (unsigned)((s->ld + 255) / 256);
    if (u_dtype == DESMO_DTYPE_BF16) {
        double* part;
        int rc = qsums_begin(qsums, grid, &part, st);
        if (rc) return rc;
        __nv_bfloat16* Ub = static_cast<__nv_bfloat16*>(U);
        if (v_dtype == DESMO_DTYPE_F64)
            preprocess_bf16_kernel<double><<<grid, 256, 0, st>>>((const double*)V, v_ld, s->n, s->ld, m_in, s->m, t_stride, d_in, d_use, flags,
                                                                 Ub, mean, part);
        else
            preprocess_bf16_kernel<float><<<grid, 256, 0, st>>>((const float*)V, v_ld, s->n, s->ld, m_in, s->m, t_stride, d_in, d_use, flags,
                                                                Ub, mean, part);
        DESMO_CUDA(cudaGetLastError());
        return qsums_end(qsums, grid, part, st);
    }
    float* Uf = static_cast<float*>(U);
    if (v_dtype == DESMO_DTYPE_F64)
        preprocess_kernel<double><<<grid, 256, 0, st>>>((const double*)V, v_ld, s->n, s->ld, m_in, s->m, t_stride, d_in, d_use, flags, Uf, mean);
    else
        preprocess_kernel<float><<<grid, 256, 0, st>>>((const float*)V, v_ld, s->n, s->ld, m_in, s->m, t_stride, d_in, d_use, flags, Uf, mean);
    DESMO_CUDA(cudaGetLastError());
    return DESMO_OK;
}

}  // namespace desmo
