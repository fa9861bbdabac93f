// Backward elimination by error at fixed coefficients (desmo_elimination_greedy): from the library Gram A = G^T G (K x K), F = G^T R
// (K x m, R = G W - U) and ||R||_F^2 of desmo_elimination_pass, remove one term per step, the one whose removal raises ||U - recon||^2
// the least.  Removing term k changes the error of snapshot t by
//     Delta_k(t) = -2 W_k(t) F_k(t) + A_kk W_k(t)^2 = W_k(t) (A_kk W_k(t) - 2 F_k(t)),
// and afterwards F_l(t) <- F_l(t) - A_lk W_k(t) for every remaining l.  Terms whose W row is zero change nothing and go first, in index
// order; then the argmin of sum_t Delta_k(t), ties to the lowest index.  O(K^2 m) fp64 arithmetic, U is not read.
//
// One launch per step, captured in sequence on the stream: block l updates F_l with the term chosen by the previous launch and scores
// l; the last block to arrive (an integer counter, no float atomics) takes the argmin over the K scores in a fixed order and records
// the choice for the next launch.  A cooperative launch would save the launch gaps but needs a grid barrier and a watchdog; at K in
// the hundreds a step is a few microseconds of work either way, and plain launches stay capturable and cannot hang.
#include <math.h>

#include "common.cuh"

namespace desmo {

constexpr int kElimThreads = 256;

struct ElimState {
    int kprev;          // term removed by the previous step whose F update is pending, or -1
    unsigned arrived;   // blocks of the current step that have written their score
};

// scratch head: [ElimState, 256 B][removed int32 K][nonzero int32 K][score fp64 K], each region 256-byte aligned
static size_t align256(size_t v) { return (v + 255) / 256 * 256; }
size_t elimination_greedy_scratch_bytes(int K) { return 256 + 2 * align256((size_t)K * 4) + align256((size_t)K * 8); }

__global__ void elim_init_kernel(const double* __restrict__ r2, int K, ElimState* __restrict__ stt, int* __restrict__ removed,
                                 double* __restrict__ predicted) {
    for (int k = threadIdx.x; k < K; k += blockDim.x) removed[k] = 0;
    if (threadIdx.x == 0) {
        stt->kprev = -1;
        stt->arrived = 0u;
        predicted[0] = *r2;
    }
}

__global__ void __launch_bounds__(kElimThreads) elim_step_kernel(const double* __restrict__ A, double* __restrict__ F,
                                                                 const float* __restrict__ W, int K, int m, int mld, int step,
                                                                 ElimState* stt, int* removed, int* nonzero, double* score,
                                                                 int32_t* __restrict__ order, double* __restrict__ predicted) {
    __shared__ double red_s[kElimThreads];
    __shared__ int red_k[kElimThreads], red_z[kElimThreads];
    __shared__ int is_last;
    const int l = blockIdx.x, tid = threadIdx.x;
    if (!removed[l]) {
        const int kp = stt->kprev;
        const double akl = kp >= 0 ? A[(long long)l * K + kp] : 0.0, all = A[(long long)l * K + l];
        double* Fl = F + (long long)l * mld;
        const float* Wl = W + (long long)l * mld;
        double acc = 0.0;
        int nz = 0;
        for (int t = tid; t < m; t += kElimThreads) {
            double f = Fl[t];
            if (kp >= 0) {
                f = fma(-akl, (double)W[(long long)kp * mld + t], f);
                Fl[t] = f;
            }
            const double w = (double)Wl[t];
            acc = fma(w, fma(all, w, -2.0 * f), acc);
            nz |= w != 0.0;
        }
        nz = __syncthreads_or(nz);
        red_s[tid] = acc;
        __syncthreads();
        for (int o = kElimThreads / 2; o > 0; o >>= 1) {
            if (tid < o) red_s[tid] += red_s[tid + o];
            __syncthreads();
        }
        if (tid == 0) {
            score[l] = isnan(red_s[0]) ? INFINITY : red_s[0];
            nonzero[l] = nz;
        }
    }
    if (tid == 0) {
        __threadfence();  // this block's score is visible before it is counted
        is_last = atomicAdd(&stt->arrived, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    // the last block: the lowest remaining index with a zero W row, else the remaining term of least score (lowest index on ties)
    double bs = INFINITY;
    int bk = K, bz = K;
    for (int k = tid; k < K; k += kElimThreads) {
        if (__ldcg(removed + k)) continue;
        if (!__ldcg(nonzero + k)) {
            bz = min(bz, k);
            continue;
        }
        const double sc = __ldcg(score + k);
        if (bk == K || sc < bs) { bs = sc; bk = k; }  // k increases within a thread: equal scores keep the lower index
    }
    red_s[tid] = bs;
    red_k[tid] = bk;
    red_z[tid] = bz;
    __syncthreads();
    for (int o = kElimThreads / 2; o > 0; o >>= 1) {
        if (tid < o) {
            const double s2 = red_s[tid + o];
            const int k2 = red_k[tid + o];
            if (k2 < K && (red_k[tid] == K || s2 < red_s[tid] || (s2 == red_s[tid] && k2 < red_k[tid]))) {
                red_s[tid] = s2;
                red_k[tid] = k2;
            }
            red_z[tid] = min(red_z[tid], red_z[tid + o]);
        }
        __syncthreads();
    }
    if (tid == 0) {
        const bool zero = red_z[0] < K;
        const int k = zero ? red_z[0] : red_k[0];
        order[step] = k;
        removed[k] = 1;
        predicted[step + 1] = zero ? predicted[step] : predicted[step] + red_s[0];
        stt->kprev = zero ? -1 : k;  // a zero row leaves F as it is
        stt->arrived = 0u;
    }
}

int elimination_greedy(int K, int m, int mld, const double* A, double* F, const double* r2, const float* W, int steps, int32_t* order,
                       double* predicted, void* scratch, cudaStream_t st) {
    uint8_t* base = static_cast<uint8_t*>(scratch);
    ElimState* stt = reinterpret_cast<ElimState*>(base);
    int* removed = reinterpret_cast<int*>(base + 256);
    int* nonzero = reinterpret_cast<int*>(base + 256 + align256((size_t)K * 4));
    double* score = reinterpret_cast<double*>(base + 256 + 2 * align256((size_t)K * 4));
    elim_init_kernel<<<1, kElimThreads, 0, st>>>(r2, K, stt, removed, predicted);
    DESMO_CUDA(cudaGetLastError());
    for (int s = 0; s < steps; ++s) {
        elim_step_kernel<<<K, kElimThreads, 0, st>>>(A, F, W, K, m, mld, s, stt, removed, nonzero, score, order, predicted);
        DESMO_CUDA(cudaGetLastError());
    }
    return DESMO_OK;
}

}  // namespace desmo
