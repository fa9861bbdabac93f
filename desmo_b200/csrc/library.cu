// Temporal side of the library: rows (free vectors or Fourier series) and W = diag(gates) * rows.
#include <cuda_bf16.h>

#include "common.cuh"

namespace desmo {

// torch.linspace(0, m, m)[t] as ATen evaluates it in fp32 (FCYL:485): step = m/(m-1); the first half counts up from
// the start, the second half counts down from the end.
__device__ __forceinline__ float t_point(int t, int m) {
    const float step = __fdiv_rn((float)m, (float)(m - 1));
    return (t < m / 2) ? __fmul_rn(step, (float)t) : __fsub_rn((float)m, __fmul_rn(step, (float)(m - 1 - t)));
}

// theta = ((2*pi*h) * t) / period in the reference's rounding order (FCYL:504): the python double 2*pi*h is rounded to
// fp32 when it multiplies the fp32 tensor, then an fp32 divide by the (1,)-shaped period parameter.
__device__ __forceinline__ float fourier_theta(int h, float t, float period) {
    const float two_pi_h = (float)(6.283185307179586 * (double)h);
    return __fdiv_rn(__fmul_rn(two_pi_h, t), period);
}

__device__ __forceinline__ float fourier_value(const float* __restrict__ c, int nF, float t, float period) {
    float z = c[0];  // a0 * ones_like(x)
    for (int h = 1; h <= nF; ++h) {
        const float th = fourier_theta(h, t, period);
        const float term = __fadd_rn(__fmul_rn(c[2 * h - 1], cosf(th)), __fmul_rn(c[2 * h], sinf(th)));
        z = __fadd_rn(z, term);
    }
    return z;
}

// grid = Kp blocks (one library term each), 256 threads over time.  kTimes: column t of a Fourier model is evaluated at
// t_points[t] (desmo_time_points_prepare) instead of t_point(t, m); the table is read by address at every launch.  The parameter
// comes last, so the instantiation without a table compiles to the kernel it was before the table existed.
template <bool kTimes>
__global__ void build_w_kernel(int K, int m, int mld, int nF, const float* __restrict__ gates, float* __restrict__ rows,
                               const float* __restrict__ coefs, const float* __restrict__ periods, float* __restrict__ W,
                               __nv_bfloat16* __restrict__ Wb, int Kp, int32_t* step_dev, float* l1_out,
                               const int32_t* __restrict__ active_pos, const float* __restrict__ t_points) {
    // Wb: three bf16 planes [3][32][mld] of W for the tcgen05 path (w = b1 + b2 + b3), rows >= K zero.
    // active_pos (null: every term active): an absent term has a zero W row and no share of the L1 sum.
    const int k = blockIdx.x;
    if (k == 0 && threadIdx.x < 32) {
        float s = 0.0f;
        for (int j = threadIdx.x; j < K; j += 32)
            if (!active_pos || active_pos[j] >= 0) s += fabsf(gates[j]);
        s = warp_sum(s);
        if (threadIdx.x == 0) {
            *l1_out = s;                       // L1 of the gates before this step's update (CYL:725-731)
            if (step_dev) *step_dev += 1;      // optimizer step counter t (Adamax bias correction)
        }
    }
    const float gate = (k < K && (!active_pos || active_pos[k] >= 0)) ? gates[k] : 0.0f;
    const float period = (nF > 0 && k < K) ? periods[k] : 1.0f;
    for (int t = threadIdx.x; t < mld; t += blockDim.x) {
        float w = 0.0f;
        if (k < K && t < m) {
            float z;
            if (nF > 0) {
                z = fourier_value(coefs + (size_t)k * (2 * nF + 1), nF, kTimes ? t_points[t] : t_point(t, m), period);
                rows[(size_t)k * mld + t] = z;
            } else {
                z = rows[(size_t)k * mld + t];
            }
            w = gate * z;
        }
        if (k < Kp) W[(size_t)k * mld + t] = w;
        if (Wb && k < 32) {
            const __nv_bfloat16 b1 = __float2bfloat16_rn(w);
            const float e1 = w - __bfloat162float(b1);
            const __nv_bfloat16 b2 = __float2bfloat16_rn(e1);
            const __nv_bfloat16 b3 = __float2bfloat16_rn(e1 - __bfloat162float(b2));
            Wb[(size_t)k * mld + t] = b1;
            Wb[(size_t)(32 + k) * mld + t] = b2;
            Wb[(size_t)(64 + k) * mld + t] = b3;
        }
    }
}

int build_w(const desmo_shape* s, int K, int Kp, const float* gates, float* rows, const float* coefs, const float* periods,
            float* W, float* Whi, float* Wlo, int32_t* step_dev, float* l1_out, cudaStream_t st, const int32_t* active_pos,
            const float* t_points) {
    (void)Wlo;
    const int grid = (Whi && Kp < 32) ? 32 : Kp;
    if (t_points)
        build_w_kernel<true><<<grid, 256, 0, st>>>(K, s->m, s->mld, s->nF, gates, rows, coefs, periods, W,
                                                   reinterpret_cast<__nv_bfloat16*>(Whi), Kp, step_dev, l1_out, active_pos, t_points);
    else
        build_w_kernel<false><<<grid, 256, 0, st>>>(K, s->m, s->mld, s->nF, gates, rows, coefs, periods, W,
                                                    reinterpret_cast<__nv_bfloat16*>(Whi), Kp, step_dev, l1_out, active_pos, nullptr);
    DESMO_CUDA(cudaGetLastError());
    return DESMO_OK;
}

// Instants of one build_w_at launch, passed by value (2 KB of kernel parameters): no device copy of the caller's host arrays, so the
// call needs no allocation and stays capturable.  Launch b writes columns [c0, c1) of W_out; the instants of columns c0 .. m_out-1.
struct AtBatch {
    int c0, c1, m_out, use_times;
    union { int32_t index[kAtBatch]; float time[kAtBatch]; };
};

// grid = Kp blocks (one library term each), 256 threads over the batch's columns.  Same z and gate * z as build_w_kernel at an
// instant t_point(index, m) or a given time; rows is only read.
__global__ void build_w_at_kernel(int K, int m, int mld, int nF, const float* __restrict__ gates, const float* __restrict__ rows,
                                  const float* __restrict__ coefs, const float* __restrict__ periods, int mld_out,
                                  float* __restrict__ W_out, float* __restrict__ rows_out, const AtBatch b) {
    const int k = blockIdx.x;
    const float gate = (k < K) ? gates[k] : 0.0f;
    const float period = (nF > 0 && k < K) ? periods[k] : 1.0f;
    for (int c = b.c0 + threadIdx.x; c < b.c1; c += blockDim.x) {
        float z = 0.0f, w = 0.0f;
        if (k < K && c < b.m_out) {
            const int i = c - b.c0;
            if (nF > 0) {
                const float t = b.use_times ? b.time[i] : t_point(b.index[i], m);
                z = fourier_value(coefs + (size_t)k * (2 * nF + 1), nF, t, period);
            } else {
                z = rows[(size_t)k * mld + b.index[i]];
            }
            w = gate * z;
        }
        W_out[(size_t)k * mld_out + c] = w;
        if (rows_out && k < K) rows_out[(size_t)k * mld_out + c] = z;
    }
}

int build_w_at(const desmo_shape* s, int K, int Kp, const float* gates, const float* rows, const float* coefs, const float* periods,
               int m_out, int mld_out, const int32_t* index, const float* times, float* W_out, float* rows_out, cudaStream_t st) {
    AtBatch b;
    b.m_out = m_out;
    b.use_times = times != nullptr;
    for (int c0 = 0; c0 < m_out; c0 += kAtBatch) {
        const int cnt = (m_out - c0 < kAtBatch) ? m_out - c0 : kAtBatch;
        b.c0 = c0;
        b.c1 = (c0 + cnt == m_out) ? mld_out : c0 + cnt;  // the last launch also zeroes the pad columns
        for (int i = 0; i < cnt; ++i) {
            if (times) b.time[i] = times[c0 + i];
            else b.index[i] = index[c0 + i];
        }
        build_w_at_kernel<<<Kp, 256, 0, st>>>(K, s->m, s->mld, s->nF, gates, rows, coefs, periods, mld_out, W_out, rows_out, b);
        DESMO_CUDA(cudaGetLastError());
    }
    return DESMO_OK;
}

}  // namespace desmo
