// Shared definitions for the desmo_b200 kernels (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/desmo_b200.h"

namespace desmo {

// Limits of the fused kernels (FFMA and fused tcgen05): library table passed by value in the kernel parameters, per-mode register arrays.
// Larger libraries (up to DESMO_MAX_R modes / DESMO_MAX_K terms) run on the GEMM path (gemm_path.cu), which has no such limits.
constexpr int kMaxR = 8;
constexpr int kMaxP = DESMO_MAX_P;
constexpr int kMaxK = 80;
constexpr int kMaxT = kMaxK;  // monomial columns that fit next to 3r trig columns
constexpr int kMaxPairs = kMaxR * (kMaxR + 1) / 2;
// per-CTA scalar partials (double): [0] sum r^2, [1 .. 1+r*r) Phi^T Phi, [1+r*r .. +3r) d omega
constexpr int kScal = 1 + kMaxR * kMaxR + 3 * kMaxR;
constexpr int kMaxSlots = 2048;

// Column order of POOL_DATA (CYL:376-434): idx[j][0..deg[j]) are the mode indices multiplied left to right.
// Passed by value in kernel parameters (constant bank, uniform access).
struct MonoTable {
    int8_t idx[kMaxT][kMaxP + 1];
    int8_t deg[kMaxT];
    // L_j = L_parent[j] * Phi_last[j]  (the same left-to-right product as POOL_DATA): lets the chain rule run as one reverse sweep
    uint8_t parent[kMaxT];
    int8_t last[kMaxT];
};

struct Workspace {  // device-side carve-up of the caller's workspace; computed identically on the host
    void* gemm;      // general-library path (gemm_path.cu), present when the fused tcgen05 kernel does not cover the shape
    float* Epart;    // [slots_x][Kp][mld]   (fused kernels only)
    double* Spart;   // [kMaxSlots][kScal]
    float* Dacc;     // [Kp][ld]   (only when the time axis is chunked)
    float* l1;       // [1] sum |gates| before the update
    float* tc;       // tcgen05 path scratch (bf16 planes of W)
    float* gram;     // [SMs][128*128] per-CTA partial Gram tiles (tcgen05 Gram)
    size_t bytes;
};

struct UpdateArgs {
    const float* red;   // [Kp*mld | loss | gram r*r | domega 3r]
    const float* dphi;  // [r][ld]  (apply mode: read; grads mode: completed in place with the ortho term)
    float* dphi_out;
    const float* P;
    float* phi; float* phi_m; float* phi_u;
    float* gates; float* gates_m; float* gates_u;
    float* rows; float* rows_m; float* rows_u;
    float* coefs; float* coefs_m; float* coefs_u;
    float* periods; float* periods_m; float* periods_u;
    float* omega; float* omega_m; float* omega_u;
    float* d_gates; float* d_rows; float* d_coefs; float* d_periods; float* d_omega;  // grads mode outputs
    const float* hyper;
    const int32_t* step_dev;
    const float* l1_in;
    float* losses_out;
    long long n, ld;
    double inv_nm;  // 1 / (n_global * m)
    int m, mld, r, K, Kp, nF;
    int apply;      // 1 = Adamax in place, 0 = write gradients
};

struct EvalArgs {
    const float* P;
    const float* phi;
    const float* omega;
    const float* W;
    float* out;
    long long n, ld;
    int m, mld, r, T, K;
    MonoTable mt;
};

// host-side launchers (one per translation unit)
int build_w(const desmo_shape* s, int K, int Kp, const float* gates, float* rows, const float* coefs, const float* periods,
            float* W, float* Whi, float* Wlo, int32_t* step_dev, float* l1_out, cudaStream_t st);
// U is [m][ld] in the element type u_dtype names (DESMO_DTYPE_F32 or DESMO_DTYPE_BF16; validated by the C ABI).
// supplied = true: U holds dL/drecon ([m][ld], fp32) and R := (n_global m / 2) * U instead of G W - U (desmo_recon_backward)
int fused_fp32(const desmo_shape* s, const MonoTable& mt, int T, int Kp, const void* U, int u_dtype, const float* P, const float* phi,
               const float* omega, const float* W, float* dphi, float* red, const Workspace& ws, cudaStream_t st, bool supplied = false);
int fused_tc(const desmo_shape* s, const MonoTable& mt, int T, int Kp, const void* U, int u_dtype, const float* P, const float* phi,
             const float* omega, const float* W, float* dphi, float* red, const Workspace& ws, cudaStream_t st, bool supplied = false,
             int phase = 0);
int fused_tc_supported(const desmo_shape* s, int Kp);
int tc_debug_read(uint64_t* out, int count);
int chain_rule_tables_selftest();
int chain_rule_sweep_selftest(int r, int p, const float* d_row, const float* phi_row, float* dphi_out);
int fused_event_ms(float* ms);
int fused_event_mean_ms(float* mean_ms, int* launches, int reset);
int fused_event_graph_ms(float* ms);
int fused_event_series_ms(float* out, int capacity, int* count);
void fused_event_record(int which, cudaStream_t st);
int launch_update(const UpdateArgs& a, cudaStream_t st);
int launch_plateau(desmo_plateau* st, const int32_t* step_dev, const float* losses, float* hyper, cudaStream_t stream);
int launch_reconstruct(const EvalArgs& a, cudaStream_t st);
int launch_colnorm2(const EvalArgs& a, cudaStream_t st);
int launch_term_norms(const float* g2, const float* gates, const float* rows, int T, int K, int m, int mld, int fourier_quirk, double* out,
                      cudaStream_t st);
int pod_gram_fp32(const desmo_shape* s, const void* U, int u_dtype, float* C, cudaStream_t st);
int pod_gram_tc(const desmo_shape* s, const void* U, int u_dtype, float* C, void* workspace, cudaStream_t st);
int pod_eig(int m, int r, const float* C, float* V, float* sigma, void* workspace, size_t workspace_bytes, cudaStream_t st);
int pod_project(const desmo_shape* s, const void* U, int u_dtype, const float* V, const float* sigma, float* P, cudaStream_t st);
// U is written as fp32 or, for u_dtype == DESMO_DTYPE_BF16, as bf16_rn of the fp32 value; qsums (optional, fp64 [2]) accumulates
// sum (u - q)^2 and sum u^2 over the n real points, u = the fp32 value, q = the stored one
int preprocess(const desmo_shape* s, const void* V, int v_dtype, long long v_ld, int m_in, int t_stride, int d_in, int d_use, int flags,
               void* U, int u_dtype, double* qsums, double* mean, cudaStream_t st);
// src [rows][src_ld] fp32 -> U[t0 .. t0 + rows)[ld] bf16 (round to nearest even, pad columns zeroed); qsums as above (may be NULL)
int snapshot_to_bf16(const desmo_shape* s, const float* src, long long src_ld, int t0, int rows, __nv_bfloat16* U, double* qsums,
                     cudaStream_t st);

struct Dims { int T, K, Kp; bool small; MonoTable mt; };  // small: within the fused kernels' limits (mt valid)
int count_terms(int r, int p);  // T = C(r+p, p) for 1 <= r <= DESMO_MAX_R, 0 <= p <= DESMO_MAX_P and T + 3r <= DESMO_MAX_K, else -1
struct GemmWorkspace;
size_t gemm_workspace_bytes(const desmo_shape* s, int T, int K, int Kp, uint8_t* base, GemmWorkspace* w);
int fused_gemm_path(const desmo_shape* s, int T, int K, int Kp, const void* U, int u_dtype, const float* P, const float* phi, const float* omega,
                    const float* W, float* dphi, float* red, float* Dacc, void* gemm_ws, cudaStream_t st, bool supplied);
int reconstruct_gemm_path(const desmo_shape* s, int T, int K, int Kp, const float* P, const float* phi, const float* omega, const float* W,
                          float* out, cudaStream_t st);
int colnorm2_gemm_path(const desmo_shape* s, int T, int K, const float* P, const float* phi, const float* omega, float* out_k, cudaStream_t st);
int launch_update_phi_generic(const UpdateArgs& a, cudaStream_t st);
int select_path(const desmo_shape* s, const Dims& d);  // DESMO_PATH_FP32 / _TC / _GEMM actually used, or <0 (error set)
int validate_shape(const desmo_shape* s, Dims* d);
int carve_workspace(const desmo_shape* s, const Dims& d, void* base, Workspace* ws);
bool use_tc_path(const desmo_shape* s, const Dims& d);

void set_error(const char* fmt, ...);
int check_cuda(cudaError_t e, const char* what);
int build_mono_table(int r, int p, MonoTable* mt);  // returns T or <0
int device_ok();

#define DESMO_CUDA(call)                                   \
    do {                                                   \
        int _rc = ::desmo::check_cuda((call), #call);      \
        if (_rc) return _rc;                               \
    } while (0)

// Snapshot element loads: bf16 -> fp32 is exact (the bf16 bits are the upper half of the fp32 word).
__device__ __forceinline__ float ldg_u(const float* p) { return __ldg(p); }
__device__ __forceinline__ float ldg_u(const __nv_bfloat16* p) {
    return __uint_as_float((uint32_t)__ldg(reinterpret_cast<const unsigned short*>(p)) << 16);
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// One library column of G at a point: Phi[] is read through a strided smem column (dynamic mode index).
__device__ __forceinline__ float monomial(const MonoTable& mt, int j, const float* phi_col, int stride) {
    const int deg = mt.deg[j];
    float v = 1.0f;
    for (int q = 0; q < deg; ++q) {
        const float f = phi_col[mt.idx[j][q] * stride];
        v = (q == 0) ? f : v * f;  // left-to-right products, as CYL:390-431
    }
    return v;
}

// Chain rule D (n x K, already scaled by 2/(n_global m)) -> d mse/d Phi_i, d mse/d omega, Phi^T Phi contributions of ONE point.
// phi_col / d_col / dphi_col are smem columns of this point (element i at [i*stride]).  Returns nothing; writes
// dphi_col[i] (i<r) and adds this point's d omega terms into dom[3r] (registers of the caller, static indexing
// avoided by going through smem in the callers).
__device__ __forceinline__ void chain_rule_point(const MonoTable& mt, int r, int T, const float* __restrict__ omega,
                                                 const float* phi_col, const float* d_col, float* dphi_col, float* dom_col,
                                                 int stride) {
    for (int i = 0; i < r; ++i) dphi_col[i * stride] = 0.0f;
    for (int j = 1; j < T; ++j) {  // j = 0 is the constant column
        const int deg = mt.deg[j];
        const float dj = d_col[j * stride];
        for (int pos = 0; pos < deg; ++pos) {
            float rest = 1.0f;
            for (int q = 0; q < deg; ++q)
                if (q != pos) rest *= phi_col[mt.idx[j][q] * stride];
            dphi_col[mt.idx[j][pos] * stride] += dj * rest;
        }
    }
    for (int i = 0; i < r; ++i) {
        const float ph = phi_col[i * stride];
        const float ws = omega[3 * i], wc = omega[3 * i + 1], wh = omega[3 * i + 2];
        const float ds = d_col[(T + i) * stride], dc = d_col[(T + r + i) * stride], dh = d_col[(T + 2 * r + i) * stride];
        const float cs = cosf(ws * ph);            // d sin(w phi)
        const float sn = sinf(wc * ph);            // -d cos(w phi)
        const float th = tanhf(wh * ph);
        const float sech2 = 1.0f - th * th;
        dphi_col[i * stride] += ds * ws * cs - dc * wc * sn + dh * wh * sech2;
        dom_col[(3 * i) * stride] = ds * ph * cs;
        dom_col[(3 * i + 1) * stride] = -dc * ph * sn;
        dom_col[(3 * i + 2) * stride] = dh * ph * sech2;
    }
}

}  // namespace desmo
