// extern "C" surface of libdesmo_b200.so (see include/desmo_b200.h): validation, workspace carve-up, launches.
#include <stdarg.h>
#include <string.h>

#include <vector>

#include "common.cuh"

namespace desmo {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int check_cuda(cudaError_t e, const char* what) {
    if (e == cudaSuccess) return DESMO_OK;
    set_error("CUDA error %s (%d) in %s", cudaGetErrorString(e), (int)e, what);
    return DESMO_ERR_CUDA;
}

int device_ok() {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) { cudaGetLastError(); set_error("no CUDA device: %s (desmo_b200 has no CPU fallback)", cudaGetErrorString(e)); return DESMO_ERR_CUDA; }
    int major = 0;
    e = cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
    if (e != cudaSuccess) { cudaGetLastError(); set_error("no CUDA device: %s (desmo_b200 has no CPU fallback)", cudaGetErrorString(e)); return DESMO_ERR_CUDA; }
    if (major != 10) { set_error("desmo_b200 is built for sm_100a only; device has compute capability major %d", major); return DESMO_ERR_CUDA; }
    return DESMO_OK;
}

static long long binom(int n, int k) {
    if (k > n) return 0;
    long long v = 1;
    for (int i = 1; i <= k; ++i) v = v * (n - k + i) / i;
    return v;
}

int count_terms(int r, int p) {
    if (r < 1 || r > DESMO_MAX_R || p < 0 || p > DESMO_MAX_P) return -1;
    long long T = 0;
    for (int k = 0; k <= p; ++k) {  // calculate_number_of_terms, CYL:448-455
        T += binom(r + k - 1, k);
        if (T + 3 * r > DESMO_MAX_K) return -1;
    }
    return (int)T;
}

int build_mono_table(int r, int p, MonoTable* mt) {
    if (r < 1 || r > kMaxR || p < 0 || p > kMaxP) return -1;
    long long T = 0;
    for (int k = 0; k <= p; ++k) T += binom(r + k - 1, k);  // calculate_number_of_terms, CYL:448-455
    if (T + 3 * r > kMaxK) return -1;
    if (!mt) return (int)T;
    memset(mt, 0, sizeof(*mt));
    int j = 0;
    mt->deg[j++] = 0;
    for (int d = 1; d <= p; ++d) {
        int idx[kMaxP];
        for (int q = 0; q < d; ++q) idx[q] = 0;
        while (true) {  // combinations with replacement of range(r), lexicographic == the nested loops of CYL:384-431
            mt->deg[j] = (int8_t)d;
            for (int q = 0; q < d; ++q) mt->idx[j][q] = (int8_t)idx[q];
            ++j;
            int q = d - 1;
            while (q >= 0 && idx[q] == r - 1) --q;
            if (q < 0) break;
            const int v = idx[q] + 1;
            for (int w = q; w < d; ++w) idx[w] = v;
        }
    }
    // parent links: term (i1..id) -> term (i1..i_{d-1}); terms of one degree are contiguous and lexicographic
    for (int t = 0; t < j; ++t) {
        const int dgr = mt->deg[t];
        mt->parent[t] = 0;
        mt->last[t] = dgr ? mt->idx[t][dgr - 1] : 0;
        if (dgr <= 1) continue;
        for (int u = 0; u < t; ++u) {
            if (mt->deg[u] != dgr - 1) continue;
            bool same = true;
            for (int q = 0; q < dgr - 1; ++q) same = same && (mt->idx[u][q] == mt->idx[t][q]);
            if (same) { mt->parent[t] = (uint8_t)u; break; }
        }
    }
    return j;
}

int validate_shape(const desmo_shape* s, Dims* d) {
    if (!s) { set_error("null shape"); return DESMO_ERR_ARG; }
    if (s->n < 1 || s->m < 2 || s->ld < s->n || s->ld % 128 != 0 || s->mld < s->m || s->mld % 16 != 0 || s->n_global < s->n) {
        set_error("bad shape: n=%lld ld=%lld (multiple of 128, >= n) m=%d mld=%d (multiple of 16, >= m) n_global=%lld",
                  (long long)s->n, (long long)s->ld, s->m, s->mld, (long long)s->n_global);
        return DESMO_ERR_ARG;
    }
    if (s->nF < 0 || s->nF > 64) { set_error("nF=%d outside 0..64", s->nF); return DESMO_ERR_UNSUPPORTED; }
    const int T = count_terms(s->r, s->polyorder);
    if (T < 0) {
        set_error("unsupported library: r=%d polyorder=%d (need 1<=r<=%d, 0<=p<=%d, T+3r<=%d)", s->r, s->polyorder, DESMO_MAX_R, DESMO_MAX_P,
                  DESMO_MAX_K);
        return DESMO_ERR_UNSUPPORTED;
    }
    d->T = T;
    d->K = T + 3 * s->r;
    d->Kp = (d->K + 15) / 16 * 16;
    d->small = build_mono_table(s->r, s->polyorder, &d->mt) == T;  // within the fused kernels' limits (r <= 8, K <= 80)
    if (s->path < DESMO_PATH_AUTO || s->path > DESMO_PATH_GEMM) { set_error("bad path %d", s->path); return DESMO_ERR_ARG; }
    return DESMO_OK;
}

// Which implementation runs this shape.  AUTO: the fused tcgen05 kernel where it applies (K <= 32, m <= 1024), else the GEMM path.
int select_path(const desmo_shape* s, const Dims& d) {
    const bool tc_ok = d.small && fused_tc_supported(s, d.Kp) != 0;
    switch (s->path) {
        case DESMO_PATH_AUTO: return tc_ok ? DESMO_PATH_TC : DESMO_PATH_GEMM;
        case DESMO_PATH_TC:
            if (!tc_ok) { set_error("fused tcgen05 path does not cover this shape (K=%d > 32 or mld=%d > 1024 or r=%d > 8)", d.K, s->mld, s->r); return -1; }
            return DESMO_PATH_TC;
        case DESMO_PATH_FP32:
            if (!d.small) { set_error("FFMA path covers r <= %d, K <= %d (got r=%d, K=%d)", kMaxR, kMaxK, s->r, d.K); return -1; }
            return DESMO_PATH_FP32;
        default: return DESMO_PATH_GEMM;
    }
}

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

int carve_workspace(const desmo_shape* s, const Dims& d, void* base, Workspace* ws) {
    int dev = 0, sms = 0;
    DESMO_CUDA(cudaGetDevice(&dev));
    DESMO_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    size_t off = 0;
    char* b = static_cast<char*>(base);
    const int path = select_path(s, d);
    if (path < 0) return DESMO_ERR_UNSUPPORTED;
    const bool fused = path != DESMO_PATH_GEMM;  // per-CTA partial layouts of the fused kernels
    ws->Spart = reinterpret_cast<double*>(b + off); off = align_up(off + sizeof(double) * kMaxSlots * kScal, 256);
    ws->Epart = reinterpret_cast<float*>(b + off);  off = align_up(off + (fused ? sizeof(float) * (size_t)sms * d.Kp * s->mld : 0), 256);
    ws->l1 = reinterpret_cast<float*>(b + off);     off = align_up(off + 256, 256);
    ws->tc = reinterpret_cast<float*>(b + off);     off = align_up(off + (fused ? sizeof(float) * 2 * (size_t)(d.Kp > 32 ? d.Kp : 32) * s->mld : 0), 256);  // >= 3 bf16 planes [32][mld]
    ws->gram = reinterpret_cast<float*>(b + off);   off = align_up(off + sizeof(float) * (size_t)sms * 128 * 128 + 1024, 256);  // + pace counters
    ws->Dacc = reinterpret_cast<float*>(b + off);   off = align_up(off + sizeof(float) * (size_t)d.Kp * s->ld, 256);
    off = align_up(off, 1024);
    ws->gemm = b + off;
    if (!fused) off += gemm_workspace_bytes(s, d.T, d.K, d.Kp, nullptr, nullptr);
    ws->bytes = off;
    return DESMO_OK;
}

bool use_tc_path(const desmo_shape* s, const Dims& d) { return select_path(s, d) == DESMO_PATH_TC; }

// element type of the snapshot matrix U: fp32 or bf16 storage
static int check_u_dtype(int32_t u_dtype, const char* who) {
    if (u_dtype == DESMO_DTYPE_F32 || u_dtype == DESMO_DTYPE_BF16) return DESMO_OK;
    set_error("%s: u_dtype %d is not DESMO_DTYPE_F32 (%d) or DESMO_DTYPE_BF16 (%d)", who, (int)u_dtype, DESMO_DTYPE_F32, DESMO_DTYPE_BF16);
    return DESMO_ERR_ARG;
}

}  // namespace desmo

using namespace desmo;

extern "C" {

const char* desmo_last_error(void) { return g_err; }
const char* desmo_version(void) { return "desmo_b200 0.1 (sm_100a)"; }

int32_t desmo_num_terms(int32_t r, int32_t polyorder) { return count_terms(r, polyorder); }

int32_t desmo_padded_k(int32_t r, int32_t polyorder) {
    const int T = count_terms(r, polyorder);
    return T < 0 ? -1 : (T + 3 * r + 15) / 16 * 16;
}

int desmo_plateau_step(desmo_plateau* state_dev, const int32_t* step_dev, const float* losses_dev, float* hyper_dev, void* stream) {
    if (!state_dev || !step_dev || !losses_dev || !hyper_dev) { set_error("desmo_plateau_step: null pointer"); return DESMO_ERR_ARG; }
    return launch_plateau(state_dev, step_dev, losses_dev, hyper_dev, (cudaStream_t)stream);
}

int64_t desmo_red_count(const desmo_shape* s) {
    Dims d;
    if (validate_shape(s, &d)) return -1;
    return (int64_t)d.Kp * s->mld + 1 + s->r * s->r + 3 * s->r;
}

int32_t desmo_selected_path(const desmo_shape* s) {
    Dims d;
    if (validate_shape(s, &d)) return -1;
    return select_path(s, d);
}

int desmo_workspace_bytes(const desmo_shape* s, size_t* bytes) {
    Dims d;
    int rc = validate_shape(s, &d);
    if (rc) return rc;
    if ((rc = device_ok())) return rc;
    Workspace ws;
    if ((rc = carve_workspace(s, d, nullptr, &ws))) return rc;
    if (bytes) *bytes = ws.bytes;
    return DESMO_OK;
}

int desmo_build_w(const desmo_shape* s, const float* gates, float* rows, const float* coefs, const float* periods, float* W,
                  int32_t* step_dev, void* workspace, void* stream) {
    Dims d;
    int rc = validate_shape(s, &d);
    if (rc) return rc;
    if ((rc = device_ok())) return rc;
    if (!gates || !rows || !W || !workspace || (s->nF > 0 && (!coefs || !periods))) { set_error("desmo_build_w: null pointer"); return DESMO_ERR_ARG; }
    Workspace ws;
    if ((rc = carve_workspace(s, d, workspace, &ws))) return rc;
    const bool tc = use_tc_path(s, d);
    return build_w(s, d.K, d.Kp, gates, rows, coefs, periods, W, tc ? ws.tc : nullptr, tc ? ws.tc + (size_t)d.Kp * s->mld : nullptr,
                   step_dev, ws.l1, (cudaStream_t)stream);
}

static int fused_dispatch(const desmo_shape* s, const void* U, int32_t u_dtype, const float* P, const float* phi, const float* omega,
                          const float* W, float* dphi, float* red, void* workspace, void* stream, bool supplied, const char* who,
                          int phase = 0) {
    Dims d;
    int rc = validate_shape(s, &d);
    if (rc) return rc;
    if ((rc = check_u_dtype(u_dtype, who))) return rc;
    if ((rc = device_ok())) return rc;
    if (!U || !P || !phi || !omega || !W || !dphi || !red || !workspace) { set_error("%s: null pointer", who); return DESMO_ERR_ARG; }
    Workspace ws;
    if ((rc = carve_workspace(s, d, workspace, &ws))) return rc;
    switch (select_path(s, d)) {
        case DESMO_PATH_TC: return fused_tc(s, d.mt, d.T, d.Kp, U, u_dtype, P, phi, omega, W, dphi, red, ws, (cudaStream_t)stream, supplied, phase);
        case DESMO_PATH_FP32:
            if (phase == 2) return DESMO_OK;  // the other paths do everything in the first phase
            return fused_fp32(s, d.mt, d.T, d.Kp, U, u_dtype, P, phi, omega, W, dphi, red, ws, (cudaStream_t)stream, supplied);
        case DESMO_PATH_GEMM:
            if (phase == 2) return DESMO_OK;
            return fused_gemm_path(s, d.T, d.K, d.Kp, U, u_dtype, P, phi, omega, W, dphi, red, ws.Dacc, ws.gemm, (cudaStream_t)stream, supplied);
        default: return DESMO_ERR_UNSUPPORTED;
    }
}

int desmo_fused_residual_grad(const desmo_shape* s, const float* U, const float* P, const float* phi, const float* omega,
                              const float* W, float* dphi, float* red, void* workspace, void* stream) {
    return fused_dispatch(s, U, DESMO_DTYPE_F32, P, phi, omega, W, dphi, red, workspace, stream, false, "desmo_fused_residual_grad");
}

int desmo_fused_residual_grad_begin(const desmo_shape* s, const float* U, const float* P, const float* phi, const float* omega,
                                    const float* W, float* dphi, float* red, void* workspace, void* stream) {
    return fused_dispatch(s, U, DESMO_DTYPE_F32, P, phi, omega, W, dphi, red, workspace, stream, false, "desmo_fused_residual_grad_begin", 1);
}

int desmo_fused_residual_grad_finish(const desmo_shape* s, const float* U, const float* P, const float* phi, const float* omega,
                                     const float* W, float* dphi, float* red, void* workspace, void* stream) {
    return fused_dispatch(s, U, DESMO_DTYPE_F32, P, phi, omega, W, dphi, red, workspace, stream, false, "desmo_fused_residual_grad_finish", 2);
}

int desmo_fused_residual_grad_ex(const desmo_shape* s, const void* U, int32_t u_dtype, const float* P, const float* phi,
                                 const float* omega, const float* W, float* dphi, float* red, void* workspace, void* stream) {
    return fused_dispatch(s, U, u_dtype, P, phi, omega, W, dphi, red, workspace, stream, false, "desmo_fused_residual_grad_ex");
}

int desmo_fused_residual_grad_begin_ex(const desmo_shape* s, const void* U, int32_t u_dtype, const float* P, const float* phi,
                                       const float* omega, const float* W, float* dphi, float* red, void* workspace, void* stream) {
    return fused_dispatch(s, U, u_dtype, P, phi, omega, W, dphi, red, workspace, stream, false, "desmo_fused_residual_grad_begin_ex", 1);
}

int desmo_fused_residual_grad_finish_ex(const desmo_shape* s, const void* U, int32_t u_dtype, const float* P, const float* phi,
                                        const float* omega, const float* W, float* dphi, float* red, void* workspace, void* stream) {
    return fused_dispatch(s, U, u_dtype, P, phi, omega, W, dphi, red, workspace, stream, false, "desmo_fused_residual_grad_finish_ex", 2);
}

int desmo_recon_backward(const desmo_shape* s, const float* grad_recon, const float* P, const float* phi, const float* omega,
                         const float* W, float* dphi, float* red, void* workspace, void* stream) {
    return fused_dispatch(s, grad_recon, DESMO_DTYPE_F32, P, phi, omega, W, dphi, red, workspace, stream, true, "desmo_recon_backward");
}

static int fill_update(const desmo_shape* s, const Dims& d, const Workspace& ws, UpdateArgs* a) {
    memset(a, 0, sizeof(*a));
    a->n = s->n; a->ld = s->ld; a->m = s->m; a->mld = s->mld; a->r = s->r; a->K = d.K; a->Kp = d.Kp; a->nF = s->nF;
    a->inv_nm = 1.0 / ((double)s->n_global * (double)s->m);
    a->l1_in = ws.l1;
    return DESMO_OK;
}

int desmo_adamax_update(const desmo_shape* s, const float* red, const float* dphi, const float* P, float* phi, float* phi_m,
                        float* phi_u, float* gates, float* gates_m, float* gates_u, float* rows, float* rows_m, float* rows_u,
                        float* coefs, float* coefs_m, float* coefs_u, float* periods, float* periods_m, float* periods_u,
                        float* omega, float* omega_m, float* omega_u, const float* hyper, const int32_t* step_dev,
                        float* losses_out, void* workspace, void* stream) {
    Dims d;
    int rc = validate_shape(s, &d);
    if (rc) return rc;
    if ((rc = device_ok())) return rc;
    const bool f = s->nF > 0;
    if (!red || !dphi || !P || !phi || !phi_m || !phi_u || !gates || !gates_m || !gates_u || !rows || !omega || !omega_m || !omega_u ||
        !hyper || !step_dev || !workspace || (!f && (!rows_m || !rows_u)) ||
        (f && (!coefs || !coefs_m || !coefs_u || !periods || !periods_m || !periods_u))) {
        set_error("desmo_adamax_update: null pointer");
        return DESMO_ERR_ARG;
    }
    Workspace ws;
    if ((rc = carve_workspace(s, d, workspace, &ws))) return rc;
    UpdateArgs a;
    fill_update(s, d, ws, &a);
    a.red = red; a.dphi = dphi; a.P = P; a.phi = phi; a.phi_m = phi_m; a.phi_u = phi_u;
    a.gates = gates; a.gates_m = gates_m; a.gates_u = gates_u; a.rows = rows; a.rows_m = rows_m; a.rows_u = rows_u;
    a.coefs = coefs; a.coefs_m = coefs_m; a.coefs_u = coefs_u; a.periods = periods; a.periods_m = periods_m; a.periods_u = periods_u;
    a.omega = omega; a.omega_m = omega_m; a.omega_u = omega_u; a.hyper = hyper; a.step_dev = step_dev; a.losses_out = losses_out;
    a.apply = 1;
    return launch_update(a, (cudaStream_t)stream);
}

int desmo_assemble_grads(const desmo_shape* s, const float* red, float* dphi, const float* P, const float* phi, const float* gates,
                         const float* rows, const float* coefs, const float* periods, const float* hyper, float* d_gates,
                         float* d_rows, float* d_coefs, float* d_periods, float* d_omega, float* losses_out, void* workspace,
                         void* stream) {
    Dims d;
    int rc = validate_shape(s, &d);
    if (rc) return rc;
    if ((rc = device_ok())) return rc;
    const bool f = s->nF > 0;
    if (!red || !dphi || !P || !phi || !gates || !rows || !hyper || !d_gates || !d_omega || !workspace || (!f && !d_rows) ||
        (f && (!coefs || !periods || !d_coefs || !d_periods))) {
        set_error("desmo_assemble_grads: null pointer");
        return DESMO_ERR_ARG;
    }
    Workspace ws;
    if ((rc = carve_workspace(s, d, workspace, &ws))) return rc;
    UpdateArgs a;
    fill_update(s, d, ws, &a);
    a.red = red; a.dphi = dphi; a.dphi_out = dphi; a.P = P; a.phi = const_cast<float*>(phi);
    a.gates = const_cast<float*>(gates); a.rows = const_cast<float*>(rows); a.coefs = const_cast<float*>(coefs);
    a.periods = const_cast<float*>(periods); a.hyper = hyper; a.d_gates = d_gates; a.d_rows = d_rows; a.d_coefs = d_coefs;
    a.d_periods = d_periods; a.d_omega = d_omega; a.losses_out = losses_out;
    a.apply = 0;
    return launch_update(a, (cudaStream_t)stream);
}

int desmo_reconstruct(const desmo_shape* s, const float* P, const float* phi, const float* omega, const float* W, float* out,
                      void* stream) {
    Dims d;
    int rc = validate_shape(s, &d);
    if (rc) return rc;
    if ((rc = device_ok())) return rc;
    if (!P || !phi || !omega || !W || !out) { set_error("desmo_reconstruct: null pointer"); return DESMO_ERR_ARG; }
    if (!d.small) return reconstruct_gemm_path(s, d.T, d.K, d.Kp, P, phi, omega, W, out, (cudaStream_t)stream);
    EvalArgs a{};
    a.P = P; a.phi = phi; a.omega = omega; a.W = W; a.out = out; a.n = s->n; a.ld = s->ld; a.m = s->m; a.mld = s->mld;
    a.r = s->r; a.T = d.T; a.K = d.K; a.mt = d.mt;
    return launch_reconstruct(a, (cudaStream_t)stream);
}

int desmo_library_colnorm2(const desmo_shape* s, const float* P, const float* phi, const float* omega, float* out_k, void* stream) {
    Dims d;
    int rc = validate_shape(s, &d);
    if (rc) return rc;
    if ((rc = device_ok())) return rc;
    if (!phi || !omega || !out_k) { set_error("desmo_library_colnorm2: null pointer"); return DESMO_ERR_ARG; }
    if (!d.small) return colnorm2_gemm_path(s, d.T, d.K, P, phi, omega, out_k, (cudaStream_t)stream);
    EvalArgs a{};
    a.P = P; a.phi = phi; a.omega = omega; a.out = out_k; a.n = s->n; a.ld = s->ld; a.m = s->m; a.mld = s->mld;
    a.r = s->r; a.T = d.T; a.K = d.K; a.mt = d.mt;
    return launch_colnorm2(a, (cudaStream_t)stream);
}

int desmo_term_norms(const desmo_shape* s, const float* g2, const float* gates, const float* rows, int32_t fourier_quirk,
                     double* norms_out, void* stream) {
    Dims d;
    int rc = validate_shape(s, &d);
    if (rc) return rc;
    if ((rc = device_ok())) return rc;
    if (!g2 || !gates || !rows || !norms_out) { set_error("desmo_term_norms: null pointer"); return DESMO_ERR_ARG; }
    if (fourier_quirk && d.T > s->m) { set_error("desmo_term_norms: the Fourier scripts' poly_norm reads time index i for term i: needs T <= m"); return DESMO_ERR_ARG; }
    return launch_term_norms(g2, gates, rows, d.T, d.K, s->m, s->mld, fourier_quirk, norms_out, (cudaStream_t)stream);
}

int desmo_last_fused_kernel_ms(float* ms) {
    if (!ms) { set_error("desmo_last_fused_kernel_ms: null"); return DESMO_ERR_ARG; }
    const int rc = fused_event_ms(ms);
    if (rc) set_error("desmo_last_fused_kernel_ms: no timed launch (set DESMO_KERNEL_EVENTS=1 before the first call)");
    return rc;
}

int desmo_selftest_tables(void) {
    const int n = chain_rule_tables_selftest();
    if (n < 0) set_error("desmo_selftest_tables: a compile-time monomial table differs from build_mono_table");
    return n;
}

int desmo_selftest_chain_sweep(int32_t r, int32_t polyorder, const float* d_row, const float* phi_row, float* dphi_out) {
    if (!d_row || !phi_row || !dphi_out) { set_error("desmo_selftest_chain_sweep: null pointer"); return DESMO_ERR_ARG; }
    if (chain_rule_sweep_selftest(r, polyorder, d_row, phi_row, dphi_out)) {
        set_error("desmo_selftest_chain_sweep: no compile-time chain-rule kernel for r=%d polyorder=%d", r, polyorder);
        return DESMO_ERR_UNSUPPORTED;
    }
    return DESMO_OK;
}

int desmo_fused_kernel_ms_mean(float* mean_ms, int32_t* launches, int32_t reset) {
    int n = 0;
    const int rc = fused_event_mean_ms(mean_ms, &n, reset);
    if (launches) *launches = n;
    if (rc) set_error("desmo_fused_kernel_ms_mean: CUDA event query failed");
    return rc;
}

int desmo_fused_kernel_ms_series(float* out_ms, int32_t capacity, int32_t* count) {
    if (!out_ms || capacity < 1) { set_error("desmo_fused_kernel_ms_series: bad argument"); return DESMO_ERR_ARG; }
    int n = 0;
    const int rc = fused_event_series_ms(out_ms, capacity, &n);
    if (count) *count = n;
    if (rc) set_error("desmo_fused_kernel_ms_series: CUDA event query failed");
    return rc;
}

int desmo_graph_fused_kernel_ms(float* ms) {
    if (!ms) { set_error("desmo_graph_fused_kernel_ms: null"); return DESMO_ERR_ARG; }
    const int rc = fused_event_graph_ms(ms);
    if (rc) set_error("desmo_graph_fused_kernel_ms: no captured launch was timed (DESMO_KERNEL_EVENTS=1 and one eager call before the capture)");
    return rc;
}

int desmo_debug_timers(const desmo_shape* s, void* workspace, uint64_t* out_host, int32_t count) {
    (void)s; (void)workspace;
    if (!out_host || count < 1) { set_error("desmo_debug_timers: bad argument"); return DESMO_ERR_ARG; }
    if (tc_debug_read(out_host, count)) { set_error("desmo_debug_timers: no debug run recorded (set DESMO_TC_DEBUG=1)"); return DESMO_ERR_ARG; }
    return DESMO_OK;
}

int desmo_pod_gram_ex(const desmo_shape* s, const void* U, int32_t u_dtype, float* C, void* workspace, void* stream) {
    Dims d;
    int rc = validate_shape(s, &d);
    if (rc) return rc;
    if ((rc = check_u_dtype(u_dtype, "desmo_pod_gram"))) return rc;
    if ((rc = device_ok())) return rc;
    if (!U || !C) { set_error("desmo_pod_gram: null pointer"); return DESMO_ERR_ARG; }
    if (s->path != DESMO_PATH_FP32 && workspace) {
        Workspace ws;
        if ((rc = carve_workspace(s, d, workspace, &ws))) return rc;
        rc = pod_gram_tc(s, U, u_dtype, C, ws.gram, (cudaStream_t)stream);
        if (rc != DESMO_ERR_UNSUPPORTED) return rc;  // shapes the tensor-core Gram does not cover run on the FFMA Gram kernel
    }
    return pod_gram_fp32(s, U, u_dtype, C, (cudaStream_t)stream);
}

int desmo_pod_gram(const desmo_shape* s, const float* U, float* C, void* workspace, void* stream) {
    return desmo_pod_gram_ex(s, U, DESMO_DTYPE_F32, C, workspace, stream);
}

int desmo_pod_eig(int32_t m, int32_t r, const float* C, float* V, float* sigma, void* workspace, size_t workspace_bytes, void* stream) {
    int rc = device_ok();
    if (rc) return rc;
    if (!C || !V || !sigma || !workspace || m < 2 || r < 1) { set_error("desmo_pod_eig: bad argument"); return DESMO_ERR_ARG; }
    return pod_eig(m, r, C, V, sigma, workspace, workspace_bytes, (cudaStream_t)stream);
}

int desmo_pod_project_ex(const desmo_shape* s, const void* U, int32_t u_dtype, const float* V, const float* sigma, float* P, void* stream) {
    Dims d;
    int rc = validate_shape(s, &d);
    if (rc) return rc;
    if ((rc = check_u_dtype(u_dtype, "desmo_pod_project"))) return rc;
    if ((rc = device_ok())) return rc;
    if (!U || !V || !sigma || !P) { set_error("desmo_pod_project: null pointer"); return DESMO_ERR_ARG; }
    return pod_project(s, U, u_dtype, V, sigma, P, (cudaStream_t)stream);
}

int desmo_pod_project(const desmo_shape* s, const float* U, const float* V, const float* sigma, float* P, void* stream) {
    return desmo_pod_project_ex(s, U, DESMO_DTYPE_F32, V, sigma, P, stream);
}

int desmo_snapshot_to_bf16(const desmo_shape* s, const float* src, int64_t src_ld, int32_t t0, int32_t rows, void* U, double* qsums,
                           void* stream) {
    Dims d;
    int rc = validate_shape(s, &d);
    if (rc) return rc;
    if (!src || !U) { set_error("desmo_snapshot_to_bf16: null pointer"); return DESMO_ERR_ARG; }
    if (src_ld < s->n || rows < 0 || t0 < 0 || (int64_t)t0 + rows > s->m) {
        set_error("desmo_snapshot_to_bf16: need src_ld >= n and 0 <= t0 <= t0 + rows <= m (got src_ld=%lld t0=%d rows=%d n=%lld m=%d)",
                  (long long)src_ld, t0, rows, (long long)s->n, s->m);
        return DESMO_ERR_ARG;
    }
    if ((rc = device_ok())) return rc;
    if (rows == 0) return DESMO_OK;
    return snapshot_to_bf16(s, src, src_ld, t0, rows, static_cast<__nv_bfloat16*>(U), qsums, (cudaStream_t)stream);
}

int desmo_preprocess(const desmo_shape* s, const void* V, int32_t v_dtype, int64_t v_ld, int32_t m_in, int32_t t_stride, int32_t d_in,
                     int32_t d_use, int32_t flags, float* U, double* mean, void* stream) {
    return desmo_preprocess_ex(s, V, v_dtype, v_ld, m_in, t_stride, d_in, d_use, flags, U, DESMO_DTYPE_F32, nullptr, mean, stream);
}

int desmo_preprocess_ex(const desmo_shape* s, const void* V, int32_t v_dtype, int64_t v_ld, int32_t m_in, int32_t t_stride, int32_t d_in,
                        int32_t d_use, int32_t flags, void* U, int32_t u_dtype, double* qsums, double* mean, void* stream) {
    Dims d;
    int rc = validate_shape(s, &d);
    if (rc) return rc;
    if (!V || !U) { set_error("desmo_preprocess: null pointer"); return DESMO_ERR_ARG; }
    if ((rc = check_u_dtype(u_dtype, "desmo_preprocess"))) return rc;
    if (qsums && u_dtype != DESMO_DTYPE_BF16) { set_error("desmo_preprocess: qsums needs bf16 output (fp32 output is not quantised)"); return DESMO_ERR_ARG; }
    if (v_dtype != DESMO_DTYPE_F32 && v_dtype != DESMO_DTYPE_F64) { set_error("desmo_preprocess: v_dtype must be F32 or F64"); return DESMO_ERR_ARG; }
    if (d_in < 1 || d_in > 3 || d_use < 1 || d_use > d_in) { set_error("desmo_preprocess: need 1 <= d_use <= d_in <= 3"); return DESMO_ERR_ARG; }
    if (!(flags & DESMO_PRE_MAGNITUDE) && d_in != 1) {
        set_error("desmo_preprocess: without DESMO_PRE_MAGNITUDE every component is its own row (pass n = points * d, d_in = 1)");
        return DESMO_ERR_ARG;
    }
    if (t_stride < 1 || m_in < 1 || s->m != (m_in + t_stride - 1) / t_stride) {
        set_error("desmo_preprocess: shape.m must equal ceil(m_in / t_stride)");
        return DESMO_ERR_ARG;
    }
    if (v_ld < s->n * d_in) { set_error("desmo_preprocess: v_ld < n * d_in"); return DESMO_ERR_ARG; }
    if ((rc = device_ok())) return rc;
    return preprocess(s, V, v_dtype, v_ld, m_in, t_stride, d_in, d_use, flags, U, u_dtype, qsums, mean, (cudaStream_t)stream);
}

}  // extern "C"
