// Loss assembly, regulariser sub-gradients and the Adamax update for every parameter, one launch.
//   gates/rows/omega(/coefs/periods) are replicated on every rank and updated identically from the all-reduced `red`;
//   phi is the rank's own slab.  Reference: CYL:714-733 (losses), CYL:766 (autograd of the regularisers),
//   torch.optim.Adamax (_single_tensor_adamax): m += (1-b1)(g-m); u = max(b2*u, |g|+eps); p -= lr/(1-b1^t) * m/u.
#include "common.cuh"

namespace desmo {

__device__ __forceinline__ float sgn(float v) { return (v > 0.0f) ? 1.0f : ((v < 0.0f) ? -1.0f : 0.0f); }

__device__ __forceinline__ void adamax(float* p, float* m, float* u, float g, float clr) {
    float mm = *m, uu = *u;
    mm = mm + 0.1f * (g - mm);                        // exp_avg.lerp_(grad, 1 - beta1)
    uu = fmaxf(uu * 0.999f, fabsf(g) + 1e-8f);        // max(beta2 * exp_inf, |grad| + eps)
    *m = mm;
    *u = uu;
    *p = *p - clr * mm / uu;                          // addcdiv_(exp_avg, exp_inf, value=-clr)
}

__device__ __forceinline__ float clr_of(float lr, int step) {
    const double bc = 1.0 - pow(0.9, (double)step);
    return (float)((double)lr / bc);
}

__device__ float block_sum(float v, float* sh) {  // blockDim.x == 256
    v = warp_sum(v);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
    __syncthreads();
    float s = 0.0f;
#pragma unroll
    for (int w = 0; w < 8; ++w) s += sh[w];
    return s;
}

__device__ __forceinline__ float t_point_u(int t, int m) {
    const float step = __fdiv_rn((float)m, (float)(m - 1));
    return (t < m / 2) ? __fmul_rn(step, (float)t) : __fsub_rn((float)m, __fmul_rn(step, (float)(m - 1 - t)));
}

// kTimes: the Fourier gradients take column t at a.t_points[t] (desmo_time_points_prepare) instead of t_point_u(t, m); without a
// table the instantiation is the kernel it was before the table existed (a.t_points is the last field of UpdateArgs).
template <bool kTimes>
__global__ void __launch_bounds__(256) update_kernel(const UpdateArgs a) {
    __shared__ float sh[8];
    __shared__ float gsign[kMaxR * kMaxR];
    __shared__ float cgrad[2 * 64 + 2];
    const int tid = threadIdx.x;
    const int b = blockIdx.x;
    const int step = a.apply ? *a.step_dev : 1;
    const float scale = (float)(2.0 * a.inv_nm);
    const float lam = a.hyper[DESMO_HYP_L1_LAMBDA];
    const long long eoff = (long long)a.Kp * a.mld;

    if (b < a.K) {
        // ---------------- one library term: temporal row + its gate ----------------
        const int k = b;
        if (a.active_pos && a.active_pos[k] < 0) {
            // absent from the model (active set): nothing is updated, its gradients are exactly zero
            if (!a.apply) {
                if (a.nF == 0) {
                    for (int t = tid; t < a.m; t += 256) a.d_rows[(long long)k * a.mld + t] = 0.0f;
                } else {
                    if (tid < 2 * a.nF + 1) a.d_coefs[(long long)k * (2 * a.nF + 1) + tid] = 0.0f;
                    if (tid == 0) a.d_periods[k] = 0.0f;
                }
                if (tid == 0) a.d_gates[k] = 0.0f;
            }
            return;
        }
        const float gate = a.gates[k];
        const float* E = a.red + (long long)k * a.mld;
        float* row = a.rows + (long long)k * a.mld;
        float acc = 0.0f;
        if (a.nF == 0) {
            const float clr = clr_of(a.hyper[DESMO_HYP_LR_Z], step);
            for (int t = tid; t < a.m; t += 256) {
                const float e = scale * E[t];
                acc = fmaf(row[t], e, acc);
                const float g = gate * e;
                if (a.apply) adamax(row + t, a.rows_m + (long long)k * a.mld + t, a.rows_u + (long long)k * a.mld + t, g, clr);
                else a.d_rows[(long long)k * a.mld + t] = g;
            }
        } else {
            const int nF = a.nF, width = 2 * nF + 1;
            const float period = a.periods[k];
            const float* c = a.coefs + (long long)k * width;
            float a0 = 0.0f, dper = 0.0f;
            for (int t = tid; t < a.m; t += 256) {
                const float e = scale * E[t];
                acc = fmaf(row[t], e, acc);
                a0 += gate * e;
            }
            a0 = block_sum(a0, sh);
            if (tid == 0) cgrad[0] = a0;
            for (int h = 1; h <= nF; ++h) {
                float ca = 0.0f, sa = 0.0f;
                const float two_pi_h = (float)(6.283185307179586 * (double)h);
                const float ah = c[2 * h - 1], bh = c[2 * h];
                for (int t = tid; t < a.m; t += 256) {
                    const float dz = gate * (scale * E[t]);
                    const float th = __fdiv_rn(__fmul_rn(two_pi_h, kTimes ? a.t_points[t] : t_point_u(t, a.m)), period);
                    const float cs = cosf(th), sn = sinf(th);
                    ca = fmaf(dz, cs, ca);
                    sa = fmaf(dz, sn, sa);
                    dper = fmaf(dz * (th / period), ah * sn - bh * cs, dper);  // d theta / d period = -theta / period
                }
                ca = block_sum(ca, sh);
                sa = block_sum(sa, sh);
                if (tid == 0) { cgrad[2 * h - 1] = ca; cgrad[2 * h] = sa; }
            }
            dper = block_sum(dper, sh);
            __syncthreads();
            if (tid < width) {
                if (a.apply) adamax(a.coefs + (long long)k * width + tid, a.coefs_m + (long long)k * width + tid,
                                    a.coefs_u + (long long)k * width + tid, cgrad[tid], clr_of(a.hyper[DESMO_HYP_LR_Z], step));
                else a.d_coefs[(long long)k * width + tid] = cgrad[tid];
            }
            if (tid == 0) {
                if (a.apply) adamax(a.periods + k, a.periods_m + k, a.periods_u + k, dper, clr_of(a.hyper[DESMO_HYP_LR_PERIOD], step));
                else a.d_periods[k] = dper;
            }
        }
        acc = block_sum(acc, sh);
        if (tid == 0) {
            const float g = acc + lam * sgn(gate);  // d/dgate [mse + l1_lambda * |gate|]
            if (a.apply) adamax(a.gates + k, a.gates_m + k, a.gates_u + k, g, clr_of(a.hyper[DESMO_HYP_LR_GATES], step));
            else a.d_gates[k] = g;
        }
    } else if (b == a.K) {
        // ---------------- omega + the three printed losses ----------------
        const int r = a.r;
        if (tid < 3 * r) {
            // omega[3i + b] belongs to trig term T + b r + i: frozen when that term is absent
            const bool frozen = a.active_pos && a.active_pos[a.K - 3 * r + (tid % 3) * r + tid / 3] < 0;
            const float g = a.red[eoff + 1 + r * r + tid];
            if (a.apply) {
                if (!frozen) adamax(a.omega + tid, a.omega_m + tid, a.omega_u + tid, g, clr_of(a.hyper[DESMO_HYP_LR_OMEGA], step));
            } else {
                a.d_omega[tid] = frozen ? 0.0f : g;
            }
        }
        if (tid == 0 && a.losses_out) {
            const float mse = (float)((double)a.red[eoff] * a.inv_nm);
            float ortho = 0.0f;
            for (int i = 0; i < r; ++i)
                for (int j = i + 1; j < r; ++j) ortho += fabsf(a.red[eoff + 1 + i * r + j]);
            const float l1 = *a.l1_in;
            a.losses_out[0] = mse;
            a.losses_out[1] = ortho;
            a.losses_out[2] = l1;
            a.losses_out[3] = mse + a.hyper[DESMO_HYP_BETA] * ortho + lam * l1;
        }
    } else {
        // ---------------- phi slab: ortho sub-gradient + update ----------------
        const int r = a.r;
        if (tid < r * r) {
            const int i = tid / r, j = tid % r;
            gsign[tid] = (i == j) ? 0.0f : sgn(a.red[eoff + 1 + tid]);  // d|Phi_i.Phi_j| = sign(dot)
        }
        __syncthreads();
        const float beta = a.hyper[DESMO_HYP_BETA];
        const float clr = clr_of(a.hyper[DESMO_HYP_LR_PHI], step);
        const long long nb = gridDim.x - a.K - 1;
        // four consecutive points per thread (128-bit accesses; ld is a multiple of 256 floats, so every row stays 16 B aligned);
        // the arithmetic per element is unchanged
        for (long long x = ((long long)(b - a.K - 1) * 256 + tid) * 4; x < a.n; x += nb * 256 * 4) {
            const int cnt = (a.n - x >= 4) ? 4 : (int)(a.n - x);
            float lat[kMaxR][4], pod[kMaxR][4];
#pragma unroll
            for (int i = 0; i < kMaxR; ++i) {
                if (i < r) {
                    const float4 pv = *reinterpret_cast<const float4*>(a.P + (long long)i * a.ld + x);  // pad columns exist up to ld
                    const float4 fv = *reinterpret_cast<const float4*>(a.phi + (long long)i * a.ld + x);
                    pod[i][0] = pv.x; pod[i][1] = pv.y; pod[i][2] = pv.z; pod[i][3] = pv.w;
                    lat[i][0] = fv.x * pv.x; lat[i][1] = fv.y * pv.y; lat[i][2] = fv.z * pv.z; lat[i][3] = fv.w * pv.w;
                } else {
#pragma unroll
                    for (int c = 0; c < 4; ++c) pod[i][c] = lat[i][c] = 0.0f;
                }
            }
#pragma unroll
            for (int i = 0; i < kMaxR; ++i) {
                if (i < r) {
                    const long long off = (long long)i * a.ld + x;
                    const float4 dv = *reinterpret_cast<const float4*>(a.dphi + off);
                    const float dd[4] = {dv.x, dv.y, dv.z, dv.w};
                    float g[4];
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        float o = 0.0f;
#pragma unroll
                        for (int j = 0; j < kMaxR; ++j)
                            if (j < r) o = fmaf(gsign[i * r + j], lat[j][c], o);
                        g[c] = dd[c] + beta * o * pod[i][c];
                    }
                    if (a.apply) {
                        float4 pv = *reinterpret_cast<float4*>(a.phi + off), mv = *reinterpret_cast<float4*>(a.phi_m + off),
                               uv = *reinterpret_cast<float4*>(a.phi_u + off);
                        float pp[4] = {pv.x, pv.y, pv.z, pv.w}, mm[4] = {mv.x, mv.y, mv.z, mv.w}, uu[4] = {uv.x, uv.y, uv.z, uv.w};
#pragma unroll
                        for (int c = 0; c < 4; ++c)
                            if (c < cnt) adamax(&pp[c], &mm[c], &uu[c], g[c], clr);
                        *reinterpret_cast<float4*>(a.phi + off) = make_float4(pp[0], pp[1], pp[2], pp[3]);
                        *reinterpret_cast<float4*>(a.phi_m + off) = make_float4(mm[0], mm[1], mm[2], mm[3]);
                        *reinterpret_cast<float4*>(a.phi_u + off) = make_float4(uu[0], uu[1], uu[2], uu[3]);
                    } else {
                        float4 ov = *reinterpret_cast<float4*>(a.dphi_out + off);
                        float oo[4] = {ov.x, ov.y, ov.z, ov.w};
#pragma unroll
                        for (int c = 0; c < 4; ++c)
                            if (c < cnt) oo[c] = g[c];
                        *reinterpret_cast<float4*>(a.dphi_out + off) = make_float4(oo[0], oo[1], oo[2], oo[3]);
                    }
                }
            }
        }
    }
}

// phi role for r > 8 (GEMM path): CTA tile of 128 points, Phi tile and the sign matrix of the ortho sub-gradient in shared memory.
__global__ void __launch_bounds__(128) update_phi_generic_kernel(const UpdateArgs a) {
    extern __shared__ float sm_g[];
    const int r = a.r, tid = threadIdx.x;
    float* gs = sm_g;             // [r][r]  sign(Phi_i . Phi_j), zero diagonal
    float* lat_s = sm_g + r * r;  // [r][128]
    const long long eoff = (long long)a.Kp * a.mld;
    for (int e = tid; e < r * r; e += 128) gs[e] = (e / r == e % r) ? 0.0f : sgn(a.red[eoff + 1 + e]);
    const int step = a.apply ? *a.step_dev : 1;
    const float beta = a.hyper[DESMO_HYP_BETA];
    const float clr = clr_of(a.hyper[DESMO_HYP_LR_PHI], step);
    const long long ntiles = (a.n + 127) / 128;
    for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const long long x = tile * 128 + tid;
        __syncthreads();
        for (int i = 0; i < r; ++i) lat_s[i * 128 + tid] = (x < a.n) ? a.phi[(long long)i * a.ld + x] * a.P[(long long)i * a.ld + x] : 0.0f;
        __syncthreads();
        if (x >= a.n) continue;
        for (int i = 0; i < r; ++i) {
            float o = 0.0f;
            for (int j = 0; j < r; ++j) o = fmaf(gs[i * r + j], lat_s[j * 128 + tid], o);
            const long long off = (long long)i * a.ld + x;
            const float g = a.dphi[off] + beta * o * a.P[off];
            if (a.apply) adamax(a.phi + off, a.phi_m + off, a.phi_u + off, g, clr);
            else a.dphi_out[off] = g;
        }
    }
}

int launch_update_phi_generic(const UpdateArgs& a, cudaStream_t st) {
    long long nb = (a.n + 127) / 128;
    if (nb > 148 * 8) nb = 148 * 8;
    const size_t smem = sizeof(float) * ((size_t)a.r * a.r + (size_t)a.r * 128);
    DESMO_CUDA(cudaFuncSetAttribute(update_phi_generic_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    update_phi_generic_kernel<<<(unsigned)nb, 128, smem, st>>>(a);
    DESMO_CUDA(cudaGetLastError());
    return DESMO_OK;
}

int launch_update(const UpdateArgs& a, cudaStream_t st) {
    long long nb = (a.n + 1023) / 1024;  // 4 points per thread in the phi role
    if (nb > 148 * 8) nb = 148 * 8;
    if (nb < 1) nb = 1;
    if (a.nF > 64) { set_error("update: nF > 64 not supported"); return DESMO_ERR_UNSUPPORTED; }
    if (a.r > kMaxR) {
        // the phi role of update_kernel keeps per-mode register arrays (r <= 8); larger r: its own kernel, launched FIRST because the
        // rows / gates / omega roles do not touch phi and this one reads only `red`, dphi, P, phi
        int rc = launch_update_phi_generic(a, st);
        if (rc) return rc;
        nb = 0;
    }
    if (a.t_points) update_kernel<true><<<(unsigned)(a.K + 1 + nb), 256, 0, st>>>(a);
    else update_kernel<false><<<(unsigned)(a.K + 1 + nb), 256, 0, st>>>(a);
    DESMO_CUDA(cudaGetLastError());
    return DESMO_OK;
}

// ReduceLROnPlateau.step(total_loss) on the device (torch semantics: mode 'min', threshold_mode 'rel', cooldown 0).
__global__ void plateau_kernel(desmo_plateau* st, const int32_t* step_dev, const float* losses, float* hyper) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    const int epoch = *step_dev - 1;  // the epoch whose update just ran (build_w advanced the counter at its start)
    if (epoch < 0 || epoch % st->every != 0) return;
    const double metric = (double)losses[3];
    if (metric < st->best * (1.0 - st->threshold)) {
        st->best = metric;
        st->num_bad = 0;
    } else {
        st->num_bad += 1;
    }
    if (st->num_bad > st->patience) {
        for (int i = 0; i < st->n_groups; ++i) {
            const double old = st->lrs[i];
            const double nw = fmax(old * st->factor, st->min_lr);
            if (old - nw > st->eps) {
                st->lrs[i] = nw;
                hyper[i] = (float)nw;
            }
        }
        st->num_bad = 0;
        st->reductions += 1;
    }
}

int launch_plateau(desmo_plateau* st, const int32_t* step_dev, const float* losses, float* hyper, cudaStream_t stream) {
    plateau_kernel<<<1, 32, 0, stream>>>(st, step_dev, losses, hyper);
    DESMO_CUDA(cudaGetLastError());
    return DESMO_OK;
}

}  // namespace desmo
