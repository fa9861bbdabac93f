/*
 * desmo_b200 -- C ABI of the B200-native DESMO training hot path (libdesmo_b200.so).
 *
 * The reference (amir-cardiolab/DESMO) has no FFI: its boundary is the PyTorch module surface.  Each entry point
 * below replaces a span of that surface; the cited lines are in /root/reference/DESMO/cylinder_flow/DESMO-Cylinder.py
 * ("CYL") and /root/reference/DESMO_Fourier/cylinder_flow/DESMO-Cylinder.py ("FCYL").  INTEGRATION.md shows the
 * reference-side binding (ctypes + torch custom op) a maintainer would add.
 *
 * Conventions
 *   - plain pointers and sizes only; device pointers unless the name says "host"; no torch types.
 *   - every function returns 0 on success, non-zero on error; desmo_last_error() gives the thread-local message.
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream).  Calls are stream-ordered and never
 *     synchronise, except the *_host entry points, which return after their results are in host memory.
 *   - no CPU fallback: every entry point fails (DESMO_ERR_CUDA) if no sm_100 device is usable.
 *
 * Device data layout (all fp32 except U, row pitch in elements)
 *   U      [m][ld]      snapshot matrix, time-major like the reference's `snapshot` batch (CYL:708); ld >= n, ld % 128 == 0,
 *                        columns n..ld-1 must be zero.  fp32, or bf16 through the *_ex entry points (u_dtype =
 *                        DESMO_DTYPE_BF16): the kernels widen each element exactly to fp32 and compute exactly what the fp32
 *                        entry points compute on U_q.float(); half the memory and the HBM traffic of the snapshot.
 *   P      [r][ld]      POD modes, mode-major (POD_modes[:, i] of CYL:204,538-541), zero in the padding.
 *   phi    [r][ld]      phi_list[i] (CYL:506); likewise its Adamax state exp_avg / exp_inf.
 *   gates  [K]          [c_coef (T) | sin_coef (r) | cos_coef (r) | tanh_coef (r)]              (CYL:513,524-526)
 *   rows   [K][mld]     DESMO: [z_list | zsin | zcos | ztanh] free temporal vectors, mld >= m, mld % 16 == 0 (CYL:516-521)
 *   coefs  [K][2nF+1]   DESMOFourier: Fourier coefficients of each term, periods [K]             (FCYL:527-534)
 *   omega  [3r]         reference order: omega[3i+{0,1,2}] = sin/cos/tanh frequency of mode i     (CYL:530,561-563)
 *   W      [Kp][mld]    gate_k * z_k(t), Kp = K rounded up to 16, rows K..Kp-1 zero.
 *   K = T + 3r, T = C(r+p, p).  Term order inside K: monomials in combinations_with_replacement order
 *   (POOL_DATA, CYL:376-434), then sin, cos, tanh blocks.
 */
#ifndef DESMO_B200_H
#define DESMO_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DESMO_OK 0
#define DESMO_ERR_ARG 1       /* bad shape / null pointer / misaligned pitch */
#define DESMO_ERR_UNSUPPORTED 2 /* (r, p, K, m) outside what the kernels are instantiated for */
#define DESMO_ERR_CUDA 3      /* CUDA runtime error, no device, or not sm_100 */

#define DESMO_MAX_R 64     /* modes (r_DESMO) */
#define DESMO_MAX_P 7      /* POOL_DATA supports polyorder <= 7 (CYL:376-434) */
#define DESMO_MAX_K 4096   /* library terms K = C(r+p, p) + 3r, e.g. (r, p) = (8, 3): 189, (32, 2): 657, (64, 2): 2337 */

#define DESMO_PATH_AUTO 0  /* fused tcgen05 kernel when K <= 32 and m <= 1024, else the tcgen05 GEMM path */
#define DESMO_PATH_FP32 1  /* FFMA path (K <= 80, r <= 8): independent implementation kept for cross-checks */
#define DESMO_PATH_TC 2    /* fused tcgen05 kernel (K <= 32, m <= 1024), bf16-split operands (fp32-grade accuracy) */
#define DESMO_PATH_GEMM 3  /* general libraries (any K <= DESMO_MAX_K, r <= DESMO_MAX_R): three tcgen05 GEMMs per chunk of points */

typedef struct desmo_shape {
    int64_t n;        /* mesh points owned by this rank (rows of the reference's X) */
    int64_t ld;       /* pitch of U / P / phi rows, multiple of 128 */
    int64_t n_global; /* points over all ranks: the MSE is a mean over n_global*m (CYL:722) */
    int32_t m;        /* snapshots */
    int32_t mld;      /* pitch of rows / W, multiple of 16 */
    int32_t r;        /* r_DESMO (CYL:334) */
    int32_t polyorder;/* CYL:583 */
    int32_t nF;       /* 0 = DESMO (free temporal vectors); >0 = DESMOFourier with nF harmonics (FCYL:513) */
    int32_t path;     /* DESMO_PATH_* */
} desmo_shape;

/* hyper-parameters that live in device memory so that a captured CUDA graph can be replayed while the host-side
 * ReduceLROnPlateau (CYL:614,778) changes them.  Layout of the `hyper` device array (fp32): */
enum { DESMO_HYP_LR_GATES = 0, DESMO_HYP_LR_PHI, DESMO_HYP_LR_Z, DESMO_HYP_LR_OMEGA, DESMO_HYP_LR_PERIOD,
       DESMO_HYP_BETA, DESMO_HYP_L1_LAMBDA, DESMO_HYP_COUNT };

/* layout of the reduction buffer `red` (fp32), the only thing exchanged between ranks (one NCCL all-reduce):
 *   red[0 .. Kp*mld)                 E = G^T R, unscaled                     ("dA = R^T Phi" of north_star)
 *   red[Kp*mld + 0]                  sum of squared residuals
 *   red[Kp*mld + 1 .. +r*r]          Phi^T Phi (row-major r x r)              (ortho term, CYL:714-720)
 *   red[Kp*mld + 1 + r*r .. +3r]     d mse / d omega, already scaled by 2/(n_global*m), reference order */
const char* desmo_last_error(void);
const char* desmo_version(void);

/* T = calculate_number_of_terms(r, p) (CYL:448-455); K = T + 3r; Kp = padded K.  Returns <0 if unsupported. */
int32_t desmo_num_terms(int32_t r, int32_t polyorder);
int32_t desmo_padded_k(int32_t r, int32_t polyorder);
int64_t desmo_red_count(const desmo_shape* s);            /* number of floats in `red` */
/* The implementation desmo_fused_residual_grad dispatches this shape to: DESMO_PATH_FP32 / _TC / _GEMM, or <0 if unsupported. */
int32_t desmo_selected_path(const desmo_shape* s);
int desmo_workspace_bytes(const desmo_shape* s, size_t* bytes);

/* Library evaluation, temporal side: W = diag(gates) * rows  (CYL:548 `c_coef *`, CYL:565-567 `*_coef_list[i] *`);
 * with nF > 0 first evaluates rows[k][t] = fourier_series(t_points, period_k, coefs_k) (FCYL:485-506,563,570-572)
 * into `rows`.  Also advances the device-side Adamax step counter `step_dev` by one (optimizer.step(), CYL:768). */
int desmo_build_w(const desmo_shape* s, const float* gates, float* rows, const float* coefs, const float* periods,
                  float* W, int32_t* step_dev, void* workspace, void* stream);

/* The fused pass: streams U once and produces, without materialising R = G(Phi) W - U,
 *   red    (see above; overwritten, local-rank partial)
 *   dphi   [r][ld]  d mse / d phi_list (chain rule through POOL_DATA, sin/cos/tanh and phi*POD; ortho term excluded)
 * Replaces DESMO.forward + MSELoss + the mse part of total_loss.backward() (CYL:535-576,722,766). */
int desmo_fused_residual_grad(const desmo_shape* s, const float* U, const float* P, const float* phi, const float* omega,
                              const float* W, float* dphi, float* red, void* workspace, void* stream);

/* The same pass in two halves, for multi-GPU steps that overlap the exchange with compute: after _begin returns (stream-ordered) the E
 * part of red, red[0 .. Kp*mld), is final for this rank and can be all-reduced on a side stream while _finish runs the chain rule and
 * writes dphi and the scalar tail of red ([sum r^2 | Phi^T Phi | d omega], all-reduced afterwards -- 1 + r*r + 3r floats).  On the
 * paths that have no such split (FFMA, GEMM) _begin does the whole pass and _finish is a no-op.  Same arguments as above. */
int desmo_fused_residual_grad_begin(const desmo_shape* s, const float* U, const float* P, const float* phi, const float* omega,
                                    const float* W, float* dphi, float* red, void* workspace, void* stream);
int desmo_fused_residual_grad_finish(const desmo_shape* s, const float* U, const float* P, const float* phi, const float* omega,
                                     const float* W, float* dphi, float* red, void* workspace, void* stream);

/* The three calls above for a snapshot matrix of element type u_dtype (DESMO_DTYPE_F32 or DESMO_DTYPE_BF16; anything else is
 * DESMO_ERR_ARG).  The fp32 entry points are these with DESMO_DTYPE_F32.  Path selection does not depend on u_dtype. */
int desmo_fused_residual_grad_ex(const desmo_shape* s, const void* U, int32_t u_dtype, const float* P, const float* phi,
                                 const float* omega, const float* W, float* dphi, float* red, void* workspace, void* stream);
int desmo_fused_residual_grad_begin_ex(const desmo_shape* s, const void* U, int32_t u_dtype, const float* P, const float* phi,
                                       const float* omega, const float* W, float* dphi, float* red, void* workspace, void* stream);
int desmo_fused_residual_grad_finish_ex(const desmo_shape* s, const void* U, int32_t u_dtype, const float* P, const float* phi,
                                        const float* omega, const float* W, float* dphi, float* red, void* workspace, void* stream);

/* Backward of forward()'s reconstruction for an ARBITRARY upstream gradient (what autograd runs when the reference loop does
 * `recon, _, _ = model(snapshot); loss = criterion(recon, snapshot); total_loss.backward()`, CYL:711,722,766): grad_recon[m][ld]
 * = dL/drecon in the layout of U (pad columns zero).  Same kernels and outputs as desmo_fused_residual_grad with R := (n_global *
 * m / 2) * grad_recon supplied instead of formed, so that desmo_assemble_grads / desmo_adamax_update (which apply the MSE scale
 * 2 / (n_global * m)) yield exactly dL/d(parameter).  red's "sum of squared residuals" slot is meaningless after this call. */
int desmo_recon_backward(const desmo_shape* s, const float* grad_recon, const float* P, const float* phi, const float* omega,
                         const float* W, float* dphi, float* red, void* workspace, void* stream);

/* Loss assembly + regulariser sub-gradients + Adamax (CYL:714-733,592-612,765-768) for every parameter.
 * `red` must hold the all-reduced buffer.  losses_out[4] = {mse, ortho, l1, total} of the step just taken
 * (computed from the pre-update parameters, as CYL:776-777 prints them). */
int desmo_adamax_update(const desmo_shape* s, const float* red, const float* dphi, const float* P, float* phi,
                        float* phi_m, float* phi_u, float* gates, float* gates_m, float* gates_u, float* rows,
                        float* rows_m, float* rows_u, float* coefs, float* coefs_m, float* coefs_u, float* periods,
                        float* periods_m, float* periods_u, float* omega, float* omega_m, float* omega_u,
                        const float* hyper, const int32_t* step_dev, float* losses_out, void* workspace, void* stream);

/* Gradients only (for torch.autograd users who keep their own optimizer): fills d_gates[K], d_rows[K][mld]
 * (or d_coefs / d_periods when nF > 0), d_omega[3r] and completes d_phi with the ortho term. */
int desmo_assemble_grads(const desmo_shape* s, const float* red, float* dphi, const float* P, const float* phi,
                         const float* gates, const float* rows, const float* coefs, const float* periods,
                         const float* hyper, float* d_gates, float* d_rows, float* d_coefs, float* d_periods,
                         float* d_omega, float* losses_out, void* workspace, void* stream);

/* Materialise recon (the first element of forward()'s 3-tuple, CYL:576) into out[m][ld] -- evaluation only. */
int desmo_reconstruct(const desmo_shape* s, const float* P, const float* phi, const float* omega, const float* W,
                      float* out, void* stream);

/* Post-hoc sparsification inputs: squared column norms of G (K floats, local partial -- all-reduce them across ranks).
 * P == NULL evaluates the library on the raw phi_list, which is what the reference's sweep passes to poly_norm /
 * nonlinear_norm (CYL:1192-1194; the functions, CYL:624-692, never multiply by POD_modes); P != NULL gives the columns of
 * forward()'s library (phi * POD). */
int desmo_library_colnorm2(const desmo_shape* s, const float* P, const float* phi, const float* omega, float* out_k,
                           void* stream);

/* Term norms of the post-hoc sweep in closed form, K order: norms_out[j] = |gate_j| * sqrt(g2[j]) * ||z_j||  (= torch.norm(gate_j *
 * (G_j z_j^T)), poly_norm CYL:624-647 / nonlinear_norm CYL:653-692) from the (all-reduced) g2 of desmo_library_colnorm2 and
 * the temporal rows [K][mld] (for DESMOFourier: as evaluated by desmo_build_w).  fourier_quirk != 0 reproduces the Fourier
 * scripts' poly_norm, which slices the (T, m) stack of series by columns (FCYL:652,659): polynomial term i is weighted by
 * sqrt(sum_{j<T} z_j(t_i)^2).  The active mask of a threshold is norms >= threshold && gate != 0 (CYL:1228-1238,1260-1265). */
int desmo_term_norms(const desmo_shape* s, const float* g2, const float* gates, const float* rows, int32_t fourier_quirk,
                     double* norms_out, void* stream);

/* Diagnostics, host only (no GPU needed): the chain-rule kernels specialised for common libraries carry their monomial table
 * (POOL_DATA's term order, CYL:376-434) as compile-time constants; this compares each of them with the run-time enumeration
 * desmo_count_terms / the fused kernels use.  Returns the number of tables verified (> 0) or a negative value on a mismatch. */
int desmo_selftest_tables(void);
/* ... and applies the unrolled reverse sweep of such a kernel to ONE point on the host: d_row[T] = dL/dG over the monomial columns,
 * phi_row[r] = Phi(x); dphi_out[r] = sum_j d_row[j] * dG_j/dPhi_i.  DESMO_ERR_UNSUPPORTED when (r, polyorder) has no specialised kernel. */
int desmo_selftest_chain_sweep(int32_t r, int32_t polyorder, const float* d_row, const float* phi_row, float* dphi_out);

/* Measurement: device time (CUDA events on the launching stream) of the dominant kernel of the last
 * desmo_fused_residual_grad call, recorded when DESMO_KERNEL_EVENTS is set in the environment.  Synchronous. */
int desmo_last_fused_kernel_ms(float* ms);

/* Measurement: mean device time of the dominant kernel over the eager desmo_fused_residual_grad calls since the last reset (the most
 * recent 64 at most), so that a caller can launch steps back to back without synchronising in between; reset != 0 starts a new
 * series.  Synchronous. */
int desmo_fused_kernel_ms_mean(float* mean_ms, int32_t* launches, int32_t reset);
/* ... and the per-launch durations of that series, oldest first (at most `capacity`, at most 64).  Synchronous. */
int desmo_fused_kernel_ms_series(float* out_ms, int32_t capacity, int32_t* count);

/* Measurement: device time of the dominant kernel inside the last replay of a CUDA graph that captured desmo_fused_residual_grad
 * (external event-record nodes, added when DESMO_KERNEL_EVENTS is set and one eager call preceded the capture).  Synchronous. */
int desmo_graph_fused_kernel_ms(float* ms);

/* Diagnostics: per-CTA phase timers (cycles) of the tcgen05 fused kernel, recorded when DESMO_TC_DEBUG is set in the
 * environment; 16 counters per CTA.  Synchronous. */
int desmo_debug_timers(const desmo_shape* s, void* workspace, uint64_t* out_host, int32_t count);

/* POD by the method of snapshots (replaces np.linalg.svd, CYL:197-205):
 *   gram    C[m][m] = U U^T  (local partial; tcgen05 tiles with every fp32 operand split into three bf16 planes) -- all-reduce it across ranks
 *   eig     top-r eigenpairs of C (replicated, on device): sigma[r] = sqrt(lambda), V[r][m]
 *   project P[i][x] = sum_t U[t][x] V[i][t] / sigma_i, sign-normalised so that the largest-|.| entry of V_i is positive */
int desmo_pod_gram(const desmo_shape* s, const float* U, float* C, void* workspace, void* stream);
int desmo_pod_eig(int32_t m, int32_t r, const float* C, float* V, float* sigma, void* workspace, size_t workspace_bytes,
                  void* stream);
int desmo_pod_project(const desmo_shape* s, const float* U, const float* V, const float* sigma, float* P, void* stream);
/* ... for a snapshot matrix of element type u_dtype (DESMO_DTYPE_F32 / DESMO_DTYPE_BF16).  The bf16 tcgen05 Gram feeds the stored
 * rows to the tensor core as they are (one plane, 4 instead of 24 MMAs per chunk) and equals the fp32 Gram of U_q.float(). */
int desmo_pod_gram_ex(const desmo_shape* s, const void* U, int32_t u_dtype, float* C, void* workspace, void* stream);
int desmo_pod_project_ex(const desmo_shape* s, const void* U, int32_t u_dtype, const float* V, const float* sigma, float* P, void* stream);

/* Snapshot pre-processing between the reader and POD/training, on the device (reference: numpy on the host).  V is X.T as
 * read: V[m_in][v_ld] with v_ld >= n * d_in, a point's d_in components adjacent.  Replaces convert3Dto2D_data (CYL:88-106:
 * d_in = 3, d_use = 2), convertToMagnitude (CYL:109-133, float64), subtract_mean (CYL:136-149; mean over all m_in snapshots),
 * the aneurysm scripts' 1/sqrt(m) scaling (ANEU:143), the channel script's X[:,0::2] (TURB:189: t_stride = 2, s->m =
 * ceil(m_in / t_stride)) and the X.T -> FloatTensor cast (CYL:356,708).  Output U[s->m][s->ld] (pad columns zeroed) and,
 * if mean != NULL, the fp64 temporal mean[n] (X_mean). */
#define DESMO_DTYPE_F32 0
#define DESMO_DTYPE_F64 1
#define DESMO_DTYPE_BF16 2
#define DESMO_PRE_MAGNITUDE 1
#define DESMO_PRE_SUBTRACT_MEAN 2
#define DESMO_PRE_SCALE_SQRT_M 4
int desmo_preprocess(const desmo_shape* s, const void* V, int32_t v_dtype, int64_t v_ld, int32_t m_in, int32_t t_stride,
                     int32_t d_in, int32_t d_use, int32_t flags, float* U, double* mean, void* stream);
/* ... writing U in u_dtype: DESMO_DTYPE_F32 as above, or DESMO_DTYPE_BF16 = the fp32 value rounded to nearest even once more (what
 * fp32 output followed by a bf16 cast stores).  qsums (bf16 output only, may be NULL): fp64 [2] += {sum (u - q)^2, sum u^2} over the
 * n real points and s->m snapshots, u the fp32 value and q the stored one; summed in a fixed order (reproducible). */
int desmo_preprocess_ex(const desmo_shape* s, const void* V, int32_t v_dtype, int64_t v_ld, int32_t m_in, int32_t t_stride,
                        int32_t d_in, int32_t d_use, int32_t flags, void* U, int32_t u_dtype, double* qsums, double* mean, void* stream);

/* fp32 snapshot rows -> bf16 storage: src[rows][src_ld] (device, fp32, src_ld >= n) -> U[t0 .. t0 + rows)[ld] (bf16), each value
 * rounded to nearest even (cvt.rn.bf16x2.f32, = torch's .bfloat16()), columns n..ld-1 zeroed.  Lets a caller fill a bf16 U in
 * chunks without holding an fp32 copy of the whole matrix.  qsums (may be NULL) as for desmo_preprocess_ex over these rows. */
int desmo_snapshot_to_bf16(const desmo_shape* s, const float* src, int64_t src_ld, int32_t t0, int32_t rows, void* U, double* qsums,
                           void* stream);

/* torch.optim.lr_scheduler.ReduceLROnPlateau (mode 'min', relative threshold, cooldown 0; CYL:614,776-778, ANEU:613) ON THE DEVICE:
 * the reference steps it on the host with `total_loss`, i.e. one device->host round trip per scheduler epoch.  desmo_plateau_step is
 * enqueued after desmo_adamax_update of an epoch: on epochs where (epoch % every == 0) it applies the scheduler to losses[3] and
 * writes the (possibly reduced) learning rates into hyper[0 .. n_groups) for the NEXT step -- the same point in the loop where the
 * reference's scheduler.step(total_loss) takes effect.  Learning rates are kept in fp64 like Python floats and rounded to fp32 once.
 * The state lives in device memory (initialise it on the host and copy it; read it back for checkpoints). */
typedef struct desmo_plateau {
    double best;        /* +inf initially */
    double lrs[5];      /* current learning rates (gates, phi, z, omega, period) */
    double threshold;   /* 1e-4 */
    double factor;      /* 0.1 */
    double min_lr;      /* 1e-6 */
    double eps;         /* 1e-8 */
    int32_t num_bad;
    int32_t patience;
    int32_t every;      /* scheduler cadence in epochs (1: ANEU / TURB, 10: CYL) */
    int32_t n_groups;   /* 4, or 5 for the Fourier variant */
    int32_t reductions; /* number of LR reductions so far (diagnostic) */
    int32_t pad;
} desmo_plateau;
int desmo_plateau_step(desmo_plateau* state_dev, const int32_t* step_dev, const float* losses_dev, float* hyper_dev, void* stream);

/* Multi-GPU exchange over NVLink / NVSwitch PEER MEMORY instead of NCCL (SURVEY.md section 8e; replaces the
 * torch.distributed.all_reduce a multi-GPU port of CYL:766-768 would issue on the gradients).  Every rank keeps its `red`
 * contribution in a buffer all ranks of the node have mapped, followed by a pad of 2 * world uint32 flags (zeroed once, before the
 * first step, with a barrier).  Per step: desmo_peer_begin_step (before the fused pass: waits until every peer has consumed this
 * rank's previous red) ... fused pass writes this rank's red ... desmo_peer_allreduce (signals the peers, waits for theirs, adds
 * all ranks' buffers in rank order into red_sum -- bit-identical on every rank).  Stream-ordered, CUDA-graph capturable, no host
 * synchronisation; a peer that never arrives traps after ~10 s. */
#define DESMO_MAX_PEERS 16
typedef struct desmo_peer {
    int32_t world, rank;
    const uint64_t* red_ptrs;   /* DEVICE array [world]: address (as mapped in THIS process) of every rank's red buffer */
    const uint64_t* flag_ptrs;  /* DEVICE array [world]: address of every rank's flag pad (uint32 ready[world], consumed[world]) */
    uint32_t* state;            /* DEVICE, local, 2 x uint32 zero-initialised: epoch, completion counter */
} desmo_peer;
int desmo_peer_begin_step(const desmo_peer* p, void* stream);
int desmo_peer_allreduce(const desmo_peer* p, int64_t count /* floats, multiple of 4 */, float* red_sum, void* stream);

/* Device-resident training session fed from HOST memory (one process of the reference's loop, CYL:706-778).
 * desmo_session_step_host(snapshot_host) = `snapshot = x[0].type(FloatTensor).to(device)` (CYL:708, pass NULL to keep the
 * resident copy) + forward/loss/backward/optimizer.step (CYL:711-768) + `loss.item()` (CYL:769): losses_host[4] =
 * {mse, ortho, l1, total}.  Synchronous. */
typedef struct desmo_session desmo_session;
int desmo_session_create(int64_t n, int32_t m, int32_t r, int32_t polyorder, int32_t nF, int32_t path, desmo_session** out);
/* Multi-GPU (SURVEY.md section 8e: one process per GPU, each owning a slab of n of the n_global mesh points): the session calls the
 * hook between the fused pass and the update; it must sum red_device[0..count) over all ranks in place, enqueued on `stream` (e.g.
 * ncclAllReduce, or torch.distributed.all_reduce under that stream) and return 0.  Required when n_global != n. */
typedef int (*desmo_allreduce_fn)(float* red_device, int64_t count, void* stream, void* user);
int desmo_session_create_sharded(int64_t n, int64_t n_global, int32_t m, int32_t r, int32_t polyorder, int32_t nF, int32_t path,
                                 desmo_session** out);
int desmo_session_set_allreduce(desmo_session* ss, desmo_allreduce_fn fn, void* user);
int desmo_session_destroy(desmo_session* ss);
int desmo_session_set_pod_host(desmo_session* ss, const double* pod_host /*[n][r] fp64*/);
int desmo_session_set_params_host(desmo_session* ss, const float* phi /*[r][n]*/, const float* gates /*[K]*/,
                                  const float* rows_or_coefs /*[K][m] or [K][2nF+1]*/, const float* periods /*[K] or NULL*/,
                                  const float* omega /*[3r]*/);
int desmo_session_set_hyper(desmo_session* ss, const float* lrs /*[5]*/, float beta, float l1_lambda);
int desmo_session_upload_snapshot_host(desmo_session* ss, const float* snapshot_host /*[m][n]*/);
int desmo_session_step_host(desmo_session* ss, const float* snapshot_host_or_null, float* losses_host /*[4]*/);
int desmo_session_get_params_host(desmo_session* ss, float* phi, float* gates, float* rows_or_coefs, float* periods, float* omega);

/* Reference-facing whole-run entry point with HOST buffers (what the reference's training loop CYL:706-778 does for one
 * process): uploads snapshot_host[m][n] (fp32, the reference's (m, n) batch), POD modes pod_host[n][r] (fp64, as
 * POD_analysis returns them) and the packed parameters, runs `steps` fused steps, returns the parameters and the
 * per-step losses[steps][4].  lrs[5], beta, l1_lambda as in CYL:592-612,700-701. */
int desmo_train_host(int64_t n, int32_t m, int32_t r, int32_t polyorder, int32_t nF, const float* snapshot_host,
                     const double* pod_host, float* phi_host /*[r][n]*/, float* gates_host /*[K]*/,
                     float* rows_or_coefs_host /*[K][m] or [K][2nF+1]*/, float* periods_host /*[K] or NULL*/,
                     float* omega_host /*[3r]*/, const float* lrs, float beta, float l1_lambda, int32_t steps,
                     float* losses_host /*[steps][4]*/, int32_t path);

#ifdef __cplusplus
}
#endif
#endif /* DESMO_B200_H */
