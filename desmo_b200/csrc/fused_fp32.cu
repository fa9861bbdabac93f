// Fused residual + gradient pass, FP32 FFMA path (DESMO_PATH_FP32).
//
// One pass over U (time-major [m][ld]).  A CTA owns tiles of 256 mesh points (one point per thread) and one time chunk
// [tc0, tc0+mc); it walks the chunk in slabs of 16 snapshots:
//   B1  rec[t]   = sum_k g[k] W[k][t]            g = the thread's own library row, kept in registers   (CYL:548,565-572)
//       r[t]     = rec[t] - U[t][x]               (R is never written to global memory)                 (CYL:722)
//   B2  d[k]    += r[t] W[k][t]                   d = the thread's row of dG = R W^T, in registers
//   B3  E[k][t] += sum_x G[x][k] r[x][t]          cross-thread: R slab + G tile staged in smem, E chunk resident in smem
// After the last slab the chain rule through POOL_DATA / sin / cos / tanh / (phi * POD) is applied in place (single
// chunk) or d is accumulated to Dacc for the chain-rule kernel (chunked time axis, large K*m).
#include <algorithm>
#include <cstdlib>
#include <utility>

#include "common.cuh"

namespace desmo {

constexpr int kTile = 256;  // points per CTA tile == threads
constexpr int kGS = 260;    // smem row pitch of G_s / R_s (float4-aligned, rows shift by one 16B bank group)
constexpr int kBT = 16;     // snapshots per slab

struct FusedArgs {
    const void* U;  // [m][ld] fp32, or bf16 (fused_fp32_kernel<KP, __nv_bfloat16>)
    const float* P;
    const float* phi;
    const float* omega;
    const float* W;
    float* dphi;
    float* Epart;
    double* Spart;
    float* Dacc;
    long long n, ld;
    int m, mld, r, T, K, nchunk, mc;
    int cr_stages;  // chain rule: 2 = the next tile's rows are in flight while a tile is processed, 1 = when two stages do not fit
    float scale;  // 2 / (n_global * m)
    float seed_scale;  // > 0: U holds dL/drecon and R := seed_scale * U instead of G W - U (desmo_recon_backward)
    MonoTable mt;
};

template <int KP>
struct FusedSmem {
    static constexpr int red_doubles = 8 * kScal;
    static constexpr int g_off = 0;
    static constexpr int r_off = g_off + KP * kGS;
    static constexpr int scr_off = r_off + kBT * kGS;
    static constexpr int wt_off = scr_off + 8 * kBT * KP;
    static constexpr int phi_off = wt_off + 2 * kBT * KP;
    static constexpr int dphi_off = phi_off + kMaxR * kGS;
    static constexpr int e_off = dphi_off + kMaxR * kGS;
    // chain-rule scratch dom_s[3r][kGS] aliases R_s..Wt_s, which are dead by then
    static_assert(3 * kMaxR * kGS <= phi_off - r_off, "dom_s alias does not fit");
    static size_t bytes(int mc) { return red_doubles * sizeof(double) + (size_t)(e_off + KP * mc) * sizeof(float); }
};

template <int KP, class UT>
__global__ void __launch_bounds__(kTile, 1) fused_fp32_kernel(const FusedArgs a) {
    using L = FusedSmem<KP>;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double* red_s = reinterpret_cast<double*>(smem_raw);
    float* fs = reinterpret_cast<float*>(smem_raw + L::red_doubles * sizeof(double));
    float* G_s = fs + L::g_off;      // [KP][kGS]   (re-used as D_s for the chain rule)
    float* R_s = fs + L::r_off;      // [kBT][kGS]  (R_s+scr re-used as dom_s[3r][kTile] for the chain rule)
    float* scr = fs + L::scr_off;    // [8][kBT*KP]
    float* Wt_s = fs + L::wt_off;    // [2][kBT][KP]
    float* Phi_s = fs + L::phi_off;  // [kMaxR][kGS]
    float* dPhi_s = fs + L::dphi_off;
    float* E_s = fs + L::e_off;      // [KP][mc]

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int r = a.r, T = a.T, K = a.K, mc = a.mc;
    const int tc0 = blockIdx.y * mc;
    const int tc1 = min(tc0 + mc, a.mld);
    const bool single = (a.nchunk == 1);
    const long long ntiles = (a.ld + kTile - 1) / kTile;

    for (int i = tid; i < KP * mc; i += kTile) E_s[i] = 0.0f;
    for (int i = tid; i < L::red_doubles; i += kTile) red_s[i] = 0.0;
    double loss_acc = 0.0;

    for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const long long x = tile * kTile + tid;
        const bool xin = x < a.n;
        // ---- library row of this point (CYL:538-548,565-567) ----
        for (int i = 0; i < r; ++i) {
            float v = 0.0f;
            if (x < a.ld) v = a.phi[(long long)i * a.ld + x] * a.P[(long long)i * a.ld + x];
            Phi_s[i * kGS + tid] = v;
        }
        float g[KP], d[KP];
#pragma unroll
        for (int j = 0; j < KP; ++j) {
            float v = 0.0f;
            if (j < T) {
                v = monomial(a.mt, j, Phi_s + tid, kGS);
            } else if (j < K) {
                const int b = (j - T) / r, i = (j - T) - b * r;
                const float arg = a.omega[3 * i + b] * Phi_s[i * kGS + tid];
                v = (b == 0) ? sinf(arg) : (b == 1) ? cosf(arg) : tanhf(arg);
            }
            g[j] = v;
            d[j] = 0.0f;
            G_s[j * kGS + tid] = v;
        }
        // W slab 0 of this chunk
        for (int i = tid; i < kBT * KP; i += kTile) {
            const int k = i / kBT, tt = i % kBT;
            Wt_s[tt * KP + k] = a.W[(long long)k * a.mld + tc0 + tt];
        }
        __syncthreads();

        int buf = 0;
        for (int t0 = tc0; t0 < tc1; t0 += kBT, buf ^= 1) {
            // prefetch next W slab into the other buffer (visible after this slab's barriers)
            if (t0 + kBT < tc1) {
                for (int i = tid; i < kBT * KP; i += kTile) {
                    const int k = i / kBT, tt = i % kBT;
                    Wt_s[(buf ^ 1) * kBT * KP + tt * KP + k] = a.W[(long long)k * a.mld + t0 + kBT + tt];
                }
            }
            float u[kBT];
#pragma unroll
            for (int tt = 0; tt < kBT; ++tt) {
                const int t = t0 + tt;
                u[tt] = (xin && t < a.m) ? ldg_u(static_cast<const UT*>(a.U) + (long long)t * a.ld + x) : 0.0f;
            }
            const float* Wb = Wt_s + buf * kBT * KP;
            float lsum = 0.0f;
#pragma unroll
            for (int tg = 0; tg < kBT / 4; ++tg) {
                float rec[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
                for (int kc = 0; kc < KP / 4; ++kc) {
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const float4 w = *reinterpret_cast<const float4*>(Wb + (tg * 4 + j) * KP + kc * 4);
                        rec[j] = fmaf(g[kc * 4 + 0], w.x, rec[j]);
                        rec[j] = fmaf(g[kc * 4 + 1], w.y, rec[j]);
                        rec[j] = fmaf(g[kc * 4 + 2], w.z, rec[j]);
                        rec[j] = fmaf(g[kc * 4 + 3], w.w, rec[j]);
                    }
                }
                float rr[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int t = t0 + tg * 4 + j;
                    rr[j] = (xin && t < a.m) ? (a.seed_scale > 0.0f ? a.seed_scale * u[tg * 4 + j] : rec[j] - u[tg * 4 + j]) : 0.0f;
                    lsum = fmaf(rr[j], rr[j], lsum);
                    R_s[(tg * 4 + j) * kGS + tid] = rr[j];
                }
#pragma unroll
                for (int kc = 0; kc < KP / 4; ++kc) {
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const float4 w = *reinterpret_cast<const float4*>(Wb + (tg * 4 + j) * KP + kc * 4);
                        d[kc * 4 + 0] = fmaf(rr[j], w.x, d[kc * 4 + 0]);
                        d[kc * 4 + 1] = fmaf(rr[j], w.y, d[kc * 4 + 1]);
                        d[kc * 4 + 2] = fmaf(rr[j], w.z, d[kc * 4 + 2]);
                        d[kc * 4 + 3] = fmaf(rr[j], w.w, d[kc * 4 + 3]);
                    }
                }
            }
            loss_acc += (double)lsum;
            __syncthreads();  // R_s complete

            // ---- B3: E slab partial over this warp's 32-point segment ----
            {
                const int kg = lane >> 2, tl = lane & 3, p0 = warp * 32;
                float acc[KP / 8][4];
#pragma unroll
                for (int i = 0; i < KP / 8; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) acc[i][j] = 0.0f;
#pragma unroll 2
                for (int pc = 0; pc < 8; ++pc) {
                    float4 rv[4];
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        rv[j] = *reinterpret_cast<const float4*>(R_s + (tl + 4 * j) * kGS + p0 + pc * 4);
#pragma unroll
                    for (int i = 0; i < KP / 8; ++i) {
                        const float4 gv = *reinterpret_cast<const float4*>(G_s + (kg + 8 * i) * kGS + p0 + pc * 4);
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            acc[i][j] = fmaf(gv.x, rv[j].x, acc[i][j]);
                            acc[i][j] = fmaf(gv.y, rv[j].y, acc[i][j]);
                            acc[i][j] = fmaf(gv.z, rv[j].z, acc[i][j]);
                            acc[i][j] = fmaf(gv.w, rv[j].w, acc[i][j]);
                        }
                    }
                }
#pragma unroll
                for (int i = 0; i < KP / 8; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) scr[warp * kBT * KP + (kg + 8 * i) * kBT + tl + 4 * j] = acc[i][j];
            }
            __syncthreads();  // scr complete, R_s free
            for (int o = tid; o < KP * kBT; o += kTile) {
                float s = 0.0f;
#pragma unroll
                for (int w = 0; w < 8; ++w) s += scr[w * kBT * KP + o];
                const int k = o / kBT, tt = o % kBT;
                E_s[k * mc + (t0 - tc0) + tt] += s;
            }
            // next slab's first barrier orders these scr reads before scr is rewritten
        }
        __syncthreads();  // all B3 reads of G_s done

        if (single) {
            float* D_s = G_s;
            float* dom_s = R_s;
#pragma unroll
            for (int j = 0; j < KP; ++j) D_s[j * kGS + tid] = d[j] * a.scale;
            chain_rule_point(a.mt, r, T, a.omega, Phi_s + tid, D_s + tid, dPhi_s + tid, dom_s + tid, kGS);
            for (int i = 0; i < r; ++i)
                if (x < a.ld) a.dphi[(long long)i * a.ld + x] = dPhi_s[i * kGS + tid] * a.P[(long long)i * a.ld + x];
            for (int i = 0; i < 3 * r; ++i) {
                const float v = warp_sum(xin ? dom_s[i * kGS + tid] : 0.0f);
                if (lane == 0) red_s[warp * kScal + 1 + kMaxR * kMaxR + i] += (double)v;
            }
        } else {
#pragma unroll
            for (int j = 0; j < KP; ++j)
                if (j < K && xin) atomicAdd(a.Dacc + (long long)j * a.ld + x, d[j]);
        }
        if (single) {
            for (int i = 0; i < r; ++i)
                for (int j = i; j < r; ++j) {
                    const float v = warp_sum(Phi_s[i * kGS + tid] * Phi_s[j * kGS + tid]);
                    if (lane == 0) red_s[warp * kScal + 1 + i * kMaxR + j] += (double)v;
                }
        }
        __syncthreads();  // before the next tile overwrites Phi_s / G_s
    }

    // ---- flush ----
    loss_acc = warp_sum(loss_acc);
    if (lane == 0) red_s[warp * kScal + 0] = loss_acc;
    __syncthreads();
    const int slot = blockIdx.y * gridDim.x + blockIdx.x;
    for (int i = tid; i < kScal; i += kTile) {
        double s = 0.0;
        for (int w = 0; w < 8; ++w) s += red_s[w * kScal + i];
        a.Spart[(long long)slot * kScal + i] = s;
    }
    float* Eo = a.Epart + (long long)blockIdx.x * KP * a.mld;
    const int width = tc1 - tc0;
    for (int i = tid; i < KP * width; i += kTile) {
        const int k = i / width, tt = i % width;
        Eo[(long long)k * a.mld + tc0 + tt] = E_s[k * mc + tt];
    }
}

// Chain rule: Dacc [Kp][ld] (raw dG = R W^T) -> dphi, d omega, Phi^T Phi partials.  Used by the chunked FFMA path and by the
// tensor-core path.  The monomial part is ONE reverse sweep over the library: with L_j = L_parent(j) * Phi_last(j) (exactly the
// left-to-right products of POOL_DATA, CYL:390-431), adj(L_parent) += adj(L_j) * Phi_last and dPhi_last += adj(L_j) * L_parent --
// two FMAs per term instead of a product per (term, position).
// Memory-level parallelism: every thread needs K + 2r scattered floats per point (the D rows, phi, P) and the kernel is latency-bound
// if they are requested where they are used.  All rows of the NEXT tile are therefore requested with cp.async (no registers, straight
// into the other half of a double buffer) before the current tile is processed: ~35 loads per thread stay in flight across a tile's
// arithmetic (2 CTAs per SM x 256 threads x 35 x 4 B = 72 KB per SM).
__device__ __forceinline__ void cp_async4(float* dst_smem, const float* src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((uint32_t)__cvta_generic_to_shared(dst_smem)), "l"(src) : "memory");
}
template <int R>
__global__ void __launch_bounds__(kTile) chain_rule_kernel(const FusedArgs a, int slot_base) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double* red_s = reinterpret_cast<double*>(smem_raw);
    float* fs = reinterpret_cast<float*>(smem_raw + 8 * kScal * sizeof(double));
    constexpr int r = R;
    const int T = a.T, K = T + 3 * r;
    // per-thread partial sums over all tiles of this CTA (registers; R is a template parameter so that they stay there):
    // d omega [3R] and the upper triangle of Phi^T Phi; reduced across the CTA once, after the tile loop
    float om_acc[3 * R], gr_acc[R * (R + 1) / 2];
#pragma unroll
    for (int i = 0; i < 3 * R; ++i) om_acc[i] = 0.0f;
#pragma unroll
    for (int i = 0; i < R * (R + 1) / 2; ++i) gr_acc[i] = 0.0f;
    const int stage_floats = (K + 2 * r) * kTile;  // staged per tile: D rows [K], phi [r], P [r]
    float* stage0 = fs;                            // [2][K + 2r][kTile]
    const int nst = a.cr_stages;
    float* Phi_s = fs + nst * stage_floats;        // [R][kTile]
    float* dPhi_s = Phi_s + R * kTile;             // [R][kTile]
    float* L_s = dPhi_s + R * kTile;               // [T][kTile]   library values
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int i = tid; i < 8 * kScal; i += kTile) red_s[i] = 0.0;
    const long long ntiles = (a.ld + kTile - 1) / kTile;
    auto request = [&](long long tile, int buf) {  // rows of `tile` -> stage `buf`; points beyond ld are skipped (their slots are unused)
        const long long x = tile * kTile + tid;
        float* st = stage0 + buf * stage_floats + tid;
        if (x < a.ld) {
            for (int j = 0; j < K; ++j) cp_async4(st + j * kTile, a.Dacc + (long long)j * a.ld + x);
#pragma unroll
            for (int i = 0; i < r; ++i) {
                cp_async4(st + (K + i) * kTile, a.phi + (long long)i * a.ld + x);
                cp_async4(st + (K + r + i) * kTile, a.P + (long long)i * a.ld + x);
            }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    if (nst == 2 && (long long)blockIdx.x < ntiles) request(blockIdx.x, 0);
    __syncthreads();
    int buf = 0;
    for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x, buf ^= (nst - 1)) {
        const long long x = tile * kTile + tid;
        const bool xin = x < a.n, xld = x < a.ld;
        if (nst == 2 && tile + gridDim.x < ntiles) {
            request(tile + gridDim.x, buf ^ 1);
            asm volatile("cp.async.wait_group 1;" ::: "memory");
        } else {
            if (nst == 1) request(tile, 0);
            asm volatile("cp.async.wait_group 0;" ::: "memory");
        }
        // each thread reads only what it requested itself: no barrier needed
        const float* A_in = stage0 + buf * stage_floats + tid;   // D rows of this point (raw, unscaled)
        float* A_s = stage0 + buf * stage_floats;                // reused in place as the adjoints
        float pod[R];
#pragma unroll
        for (int i = 0; i < r; ++i) {
            pod[i] = xld ? A_in[(K + r + i) * kTile] : 0.0f;
            Phi_s[i * kTile + tid] = xld ? A_in[(K + i) * kTile] * pod[i] : 0.0f;
            dPhi_s[i * kTile + tid] = 0.0f;
        }
        L_s[tid] = 1.0f;
        for (int j = 1; j < T; ++j) {
            const float f = Phi_s[a.mt.last[j] * kTile + tid];
            L_s[j * kTile + tid] = (a.mt.deg[j] == 1) ? f : L_s[a.mt.parent[j] * kTile + tid] * f;
        }
        for (int j = 0; j < T; ++j) A_s[j * kTile + tid] = xin ? A_in[j * kTile] * a.scale : 0.0f;
        for (int j = T - 1; j >= 1; --j) {
            const float adj = A_s[j * kTile + tid];
            const int par = a.mt.parent[j], v = a.mt.last[j];
            dPhi_s[v * kTile + tid] = fmaf(adj, L_s[par * kTile + tid], dPhi_s[v * kTile + tid]);
            if (par > 0) A_s[par * kTile + tid] = fmaf(adj, Phi_s[v * kTile + tid], A_s[par * kTile + tid]);
        }
#pragma unroll
        for (int i = 0; i < r; ++i) {
            const float ph = Phi_s[i * kTile + tid];
            const float ws = a.omega[3 * i], wc = a.omega[3 * i + 1], wh = a.omega[3 * i + 2];
            float ds = 0.0f, dc = 0.0f, dh = 0.0f;
            if (xin) {
                ds = A_in[(T + i) * kTile] * a.scale;
                dc = A_in[(T + r + i) * kTile] * a.scale;
                dh = A_in[(T + 2 * r + i) * kTile] * a.scale;
            }
            const float cs = cosf(ws * ph), sn = sinf(wc * ph), th = tanhf(wh * ph);
            const float sech2 = 1.0f - th * th;
            const float dphi_i = dPhi_s[i * kTile + tid] + (ds * ws * cs - dc * wc * sn + dh * wh * sech2);
            if (xld) a.dphi[(long long)i * a.ld + x] = dphi_i * pod[i];
            om_acc[3 * i] += ds * ph * cs;
            om_acc[3 * i + 1] -= dc * ph * sn;
            om_acc[3 * i + 2] += dh * ph * sech2;
        }
        {
            int g = 0;
#pragma unroll
            for (int i = 0; i < r; ++i)
#pragma unroll
                for (int j = i; j < r; ++j, ++g) gr_acc[g] = fmaf(Phi_s[i * kTile + tid], Phi_s[j * kTile + tid], gr_acc[g]);
        }
    }
#pragma unroll
    for (int i = 0; i < 3 * R; ++i) {
        const float v = warp_sum(om_acc[i]);
        if (lane == 0) red_s[warp * kScal + 1 + kMaxR * kMaxR + i] += (double)v;
    }
    {
        int g = 0;
#pragma unroll
        for (int i = 0; i < r; ++i)
#pragma unroll
            for (int j = i; j < r; ++j, ++g) {
                const float v = warp_sum(gr_acc[g]);
                if (lane == 0) red_s[warp * kScal + 1 + i * kMaxR + j] += (double)v;
            }
    }
    __syncthreads();
    for (int i = tid; i < kScal; i += kTile) {
        double s = 0.0;
        for (int w = 0; w < 8; ++w) s += red_s[w * kScal + i];
        a.Spart[(long long)(slot_base + blockIdx.x) * kScal + i] = s;
    }
}
// ---- register-resident chain rule for the common small libraries ------------------------------------------------------------
// The kernel above walks the monomial table with run-time indices, so every value lives in shared memory and each step of the
// sweep is a dependent shared-memory round trip: at the headline shape it is latency-bound (210 us for 441 MB).  For a library known
// at compile time the table folds into the instruction stream: D row, library values and adjoints stay in registers, the K + 2r
// loads of a point are issued up front, the sweep is straight-line FMAs in the SAME order as above.  The table is generated at
// compile time by the enumeration of build_mono_table (capi.cu) and compared with the run-time table on the host before the launch.
template <int R, int P>
struct CtMono {
    static constexpr int count() {
        int t = 0;
        for (int k = 0; k <= P; ++k) {
            long long v = 1;
            for (int i = 1; i <= k; ++i) v = v * (R - 1 + i) / i;
            t += (int)v;
        }
        return t;
    }
    static constexpr int T = count();
    int parent[T];
    int last[T];
    int deg[T];
    constexpr CtMono() : parent{}, last{}, deg{} {
        int idxs[T][P > 0 ? P : 1] = {};
        int j = 1;
        for (int d = 1; d <= P; ++d) {
            int idx[P > 0 ? P : 1] = {};
            while (true) {
                deg[j] = d;
                for (int q = 0; q < d; ++q) idxs[j][q] = idx[q];
                ++j;
                int q = d - 1;
                while (q >= 0 && idx[q] == R - 1) --q;
                if (q < 0) break;
                const int v = idx[q] + 1;
                for (int w = q; w < d; ++w) idx[w] = v;
            }
        }
        for (int t = 0; t < T; ++t) {
            const int dg = deg[t];
            last[t] = dg ? idxs[t][dg - 1] : 0;
            if (dg <= 1) continue;
            for (int u = 0; u < t; ++u) {
                if (deg[u] != dg - 1) continue;
                bool same = true;
                for (int q = 0; q < dg - 1; ++q) same = same && (idxs[u][q] == idxs[t][q]);
                if (same) { parent[t] = u; break; }
            }
        }
    }
};
template <int R, int P>
inline constexpr CtMono<R, P> kCtMono{};

template <int... Is, class F>
__host__ __device__ __forceinline__ void static_for_impl(std::integer_sequence<int, Is...>, F&& f) {
    (f(std::integral_constant<int, Is>{}), ...);
}
template <int N, class F>
__host__ __device__ __forceinline__ void static_for(F&& f) {
    static_for_impl(std::make_integer_sequence<int, N>{}, f);
}

// Monomial part of the chain rule for ONE point, fully unrolled over the compile-time table: forward L_j = L_parent(j) * Phi_last(j)
// (POOL_DATA's left-to-right products, CYL:390-431), then the reverse sweep  dPhi_last += adj_j * L_parent,  adj_parent += adj_j * Phi_last.
// A[0..T) holds the adjoints dL/dG_j on entry and is clobbered.  Host-callable so that the CPU suite can check the unrolled code
// against the oracle (desmo_selftest_chain_sweep); on the device everything is registers.
template <int R, int P, int NA>
__host__ __device__ __forceinline__ void chain_sweep_ct(float (&A)[NA], const float (&Phi)[R], float (&dPhi)[R]) {
    constexpr int T = CtMono<R, P>::T;
    static_assert(NA >= T, "adjoint array shorter than the library");
    float L[T];
    L[0] = 1.0f;
    static_for<T - 1>([&](auto jc) {
        constexpr int j = decltype(jc)::value + 1;
        constexpr int par = kCtMono<R, P>.parent[j], v = kCtMono<R, P>.last[j], dg = kCtMono<R, P>.deg[j];
        if constexpr (dg == 1) L[j] = Phi[v];
        else L[j] = L[par] * Phi[v];
    });
    static_for<T - 1>([&](auto jc) {
        constexpr int j = T - 1 - decltype(jc)::value;
        constexpr int par = kCtMono<R, P>.parent[j], v = kCtMono<R, P>.last[j];
        const float adj = A[j];
        dPhi[v] = fmaf(adj, L[par], dPhi[v]);
        if constexpr (par > 0) A[par] = fmaf(adj, Phi[v], A[par]);
    });
}

constexpr int kCrTile = 256;  // points per CTA tile == threads (the engine pads ld to a multiple of 256; other ld: table-driven kernel)
template <int R, int P>
__global__ void __launch_bounds__(kCrTile, 2) chain_rule_reg_kernel(const FusedArgs a, int slot_base) {
    constexpr int T = CtMono<R, P>::T, K = T + 3 * R, NG = R * (R + 1) / 2, NS = 3 * R + NG;
    __shared__ double red_s[kCrTile / 32][NS];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    float om_acc[3 * R], gr_acc[NG];
#pragma unroll
    for (int i = 0; i < 3 * R; ++i) om_acc[i] = 0.0f;
#pragma unroll
    for (int i = 0; i < NG; ++i) gr_acc[i] = 0.0f;
    const long long ntiles = a.ld / kCrTile;
    for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const long long x = tile * kCrTile + tid;
        const bool xin = x < a.n;
        float A[K], ph[R], pod[R];
#pragma unroll
        for (int j = 0; j < K; ++j) A[j] = __ldcs(a.Dacc + (long long)j * a.ld + x);  // D is read exactly once
#pragma unroll
        for (int i = 0; i < R; ++i) {
            ph[i] = __ldg(a.phi + (long long)i * a.ld + x);
            pod[i] = __ldg(a.P + (long long)i * a.ld + x);
        }
        float Phi[R], dPhi[R];
#pragma unroll
        for (int i = 0; i < R; ++i) {
            Phi[i] = ph[i] * pod[i];
            dPhi[i] = 0.0f;
        }
#pragma unroll
        for (int j = 0; j < K; ++j) A[j] = xin ? A[j] * a.scale : 0.0f;
        chain_sweep_ct<R, P>(A, Phi, dPhi);
#pragma unroll
        for (int i = 0; i < R; ++i) {
            const float p_i = Phi[i];
            const float ws = a.omega[3 * i], wc = a.omega[3 * i + 1], wh = a.omega[3 * i + 2];
            const float ds = A[T + i], dc = A[T + R + i], dh = A[T + 2 * R + i];
            const float cs = cosf(ws * p_i), sn = sinf(wc * p_i), th = tanhf(wh * p_i);
            const float sech2 = 1.0f - th * th;
            const float dphi_i = dPhi[i] + (ds * ws * cs - dc * wc * sn + dh * wh * sech2);
            a.dphi[(long long)i * a.ld + x] = dphi_i * pod[i];
            om_acc[3 * i] += ds * p_i * cs;
            om_acc[3 * i + 1] -= dc * p_i * sn;
            om_acc[3 * i + 2] += dh * p_i * sech2;
        }
        {
            int g = 0;
#pragma unroll
            for (int i = 0; i < R; ++i)
#pragma unroll
                for (int j = i; j < R; ++j, ++g) gr_acc[g] = fmaf(Phi[i], Phi[j], gr_acc[g]);
        }
    }
#pragma unroll
    for (int i = 0; i < 3 * R; ++i) {
        const float v = warp_sum(om_acc[i]);
        if (lane == 0) red_s[warp][i] = (double)v;
    }
#pragma unroll
    for (int g = 0; g < NG; ++g) {
        const float v = warp_sum(gr_acc[g]);
        if (lane == 0) red_s[warp][3 * R + g] = (double)v;
    }
    __syncthreads();
    // the slot in the layout reduce_partials_kernel sums: [loss | Phi^T Phi (kMaxR x kMaxR, upper triangle) | d omega]
    double* out = a.Spart + (long long)(slot_base + blockIdx.x) * kScal;
    for (int i = tid; i < kScal; i += kCrTile) {
        int src = -1;
        if (i >= 1 + kMaxR * kMaxR && i < 1 + kMaxR * kMaxR + 3 * R) src = i - (1 + kMaxR * kMaxR);
        else if (i >= 1 && i < 1 + kMaxR * kMaxR) {
            const int gi = (i - 1) / kMaxR, gj = (i - 1) % kMaxR;
            if (gi < R && gj < R && gj >= gi) src = 3 * R + (gi * R - gi * (gi - 1) / 2 + (gj - gi));
        }
        double sum = 0.0;
        if (src >= 0)
            for (int w = 0; w < kCrTile / 32; ++w) sum += red_s[w][src];
        out[i] = sum;
    }
}
template <int R, int P>
static bool ct_table_matches(const FusedArgs& a) {
    constexpr int T = CtMono<R, P>::T;
    if (a.r != R || a.T != T) return false;
    for (int j = 1; j < T; ++j)
        if (a.mt.parent[j] != kCtMono<R, P>.parent[j] || a.mt.last[j] != kCtMono<R, P>.last[j] || a.mt.deg[j] != kCtMono<R, P>.deg[j]) return false;
    return true;
}
template <int R, int P>
static bool chain_rule_reg_try(const FusedArgs& a, int slot_base, int sms, int* nslots, cudaStream_t st, cudaError_t* err) {
    if (!ct_table_matches<R, P>(a)) return false;
    const long long ntiles = a.ld / kCrTile;
    const long long cap = (long long)sms * 2;  // 94 registers at r4p2: two CTAs of 256 threads per SM (few slots: the partial reduction walks them all)
    const int gc = (int)(ntiles < cap ? ntiles : cap);
    chain_rule_reg_kernel<R, P><<<gc, kCrTile, 0, st>>>(a, slot_base);
    *err = cudaGetLastError();
    *nslots = gc;
    return true;
}
template <int R, int P>
static int ct_table_selfcheck() {  // host only: the compile-time table against the run-time enumeration of capi.cu
    FusedArgs a{};
    a.r = R;
    a.T = build_mono_table(R, P, &a.mt);
    return ct_table_matches<R, P>(a) ? 1 : 0;
}
int chain_rule_tables_selftest() {  // number of compile-time libraries verified, or -1 on a mismatch
    const int ok = ct_table_selfcheck<4, 2>() + ct_table_selfcheck<2, 2>() + ct_table_selfcheck<2, 3>() + ct_table_selfcheck<2, 4>() +
                   ct_table_selfcheck<3, 2>() + ct_table_selfcheck<3, 3>();
    return ok == 6 ? ok : -1;
}
template <int R, int P>
static bool chain_sweep_host_try(int r, int p, const float* d_row, const float* phi_row, float* dphi_out) {
    if (r != R || p != P) return false;
    constexpr int T = CtMono<R, P>::T;
    float A[T], Phi[R], dPhi[R];
    for (int j = 0; j < T; ++j) A[j] = d_row[j];
    for (int i = 0; i < R; ++i) { Phi[i] = phi_row[i]; dPhi[i] = 0.0f; }
    chain_sweep_ct<R, P>(A, Phi, dPhi);
    for (int i = 0; i < R; ++i) dphi_out[i] = dPhi[i];
    return true;
}
// host only: the unrolled sweep of the specialised kernels applied to one point; 0 when (r, p) has a compile-time kernel
int chain_rule_sweep_selftest(int r, int p, const float* d_row, const float* phi_row, float* dphi_out) {
    return (chain_sweep_host_try<4, 2>(r, p, d_row, phi_row, dphi_out) || chain_sweep_host_try<2, 2>(r, p, d_row, phi_row, dphi_out) ||
            chain_sweep_host_try<2, 3>(r, p, d_row, phi_row, dphi_out) || chain_sweep_host_try<2, 4>(r, p, d_row, phi_row, dphi_out) ||
            chain_sweep_host_try<3, 2>(r, p, d_row, phi_row, dphi_out) || chain_sweep_host_try<3, 3>(r, p, d_row, phi_row, dphi_out)) ? 0 : 1;
}
// the libraries the fused tcgen05 kernel covers most often (K <= 32): r4p2 (headline), r2p2, r2p3, r2p4, r3p2, r3p3
static bool chain_rule_reg_dispatch(const FusedArgs& a, int slot_base, int sms, int* nslots, cudaStream_t st, cudaError_t* err) {
    static const bool off = getenv("DESMO_CHAIN_RULE_GENERIC") != nullptr;  // A/B switch: force the table-driven kernel
    if (off || a.ld % kCrTile != 0 || slot_base + sms * 2 > kMaxSlots) return false;
    return chain_rule_reg_try<4, 2>(a, slot_base, sms, nslots, st, err) || chain_rule_reg_try<2, 2>(a, slot_base, sms, nslots, st, err) ||
           chain_rule_reg_try<2, 3>(a, slot_base, sms, nslots, st, err) || chain_rule_reg_try<2, 4>(a, slot_base, sms, nslots, st, err) ||
           chain_rule_reg_try<3, 2>(a, slot_base, sms, nslots, st, err) || chain_rule_reg_try<3, 3>(a, slot_base, sms, nslots, st, err);
}

// chain_rule_kernel<R> for R = a.r (1..kMaxR)
template <int R>
static cudaError_t chain_rule_go(const FusedArgs& a, int slot_base, int gc, size_t sm, cudaStream_t st) {
    cudaError_t e = cudaFuncSetAttribute(chain_rule_kernel<R>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
    if (e != cudaSuccess) return e;
    chain_rule_kernel<R><<<gc, kTile, sm, st>>>(a, slot_base);
    return cudaGetLastError();
}
static size_t chain_rule_smem(const FusedArgs& a, int stages) {
    return 8 * kScal * sizeof(double) + (size_t)(stages * (a.T + 5 * a.r) + 2 * a.r + a.T) * kTile * sizeof(float);
}
static cudaError_t chain_rule_dispatch(const FusedArgs& a0, int slot_base, int gc, size_t, cudaStream_t st) {
    FusedArgs a = a0;
    a.cr_stages = chain_rule_smem(a0, 2) <= 110 * 1024 ? 2 : 1;  // two CTAs per SM with both stages, else one stage
    const size_t sm = chain_rule_smem(a, a.cr_stages);
    switch (a.r) {
        case 1: return chain_rule_go<1>(a, slot_base, gc, sm, st);
        case 2: return chain_rule_go<2>(a, slot_base, gc, sm, st);
        case 3: return chain_rule_go<3>(a, slot_base, gc, sm, st);
        case 4: return chain_rule_go<4>(a, slot_base, gc, sm, st);
        case 5: return chain_rule_go<5>(a, slot_base, gc, sm, st);
        case 6: return chain_rule_go<6>(a, slot_base, gc, sm, st);
        case 7: return chain_rule_go<7>(a, slot_base, gc, sm, st);
        default: return chain_rule_go<8>(a, slot_base, gc, sm, st);
    }
}

// Deterministic second stage: sum the per-CTA partials in a fixed order into `red`.
// 32 outputs per CTA, 8 warps: warp w sums the partials b = w, w+8, ... of 32 consecutive outputs (coalesced), the eight sums are
// added in warp order -- a fixed order, so the result does not depend on scheduling.
// what: 1 = the E part only, 2 = the scalar tail only (one CTA), 3 = both.  The split lets a multi-GPU step all-reduce E on a side
// stream while the chain-rule kernel is still producing the scalars (desmo_fused_residual_grad_begin / _finish).
__global__ void __launch_bounds__(256) reduce_partials_kernel(const float* __restrict__ Epart, int nx, long long ecount,
                                                              const double* __restrict__ Spart, int nslots, int r, float* __restrict__ red,
                                                              int what) {
    // E: a CTA owns 128 consecutive outputs (one float4 per lane); warp w adds the partials b = w, w + 8, ... four at a time (four
    // independent 512 B loads in flight per warp), then the eight warp sums are added in warp order.  The partials were just written
    // by the fused kernel and sit in L2: the kernel is latency-bound, hence the wide, batched loads.  ecount is a multiple of 4.
    __shared__ float4 part_s[8][32];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const long long o = ((long long)blockIdx.x * 32 + lane) * 4;
    if (what & 1) {
        float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
        if (o < ecount) {
            const float4* src = reinterpret_cast<const float4*>(Epart + o);
            const long long stride = ecount / 4;
            int b = w;
            for (; b + 24 < nx; b += 32) {
                const float4 v0 = __ldcg(src + (long long)b * stride), v1 = __ldcg(src + (long long)(b + 8) * stride);
                const float4 v2 = __ldcg(src + (long long)(b + 16) * stride), v3 = __ldcg(src + (long long)(b + 24) * stride);
                s.x = (((s.x + v0.x) + v1.x) + v2.x) + v3.x; s.y = (((s.y + v0.y) + v1.y) + v2.y) + v3.y;
                s.z = (((s.z + v0.z) + v1.z) + v2.z) + v3.z; s.w = (((s.w + v0.w) + v1.w) + v2.w) + v3.w;
            }
            for (; b < nx; b += 8) {
                const float4 v = __ldcg(src + (long long)b * stride);
                s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
            }
        }
        part_s[w][lane] = s;
        __syncthreads();
        if (w == 0 && o < ecount) {
            float4 t = part_s[0][lane];
#pragma unroll
            for (int k = 1; k < 8; ++k) { const float4 v = part_s[k][lane]; t.x += v.x; t.y += v.y; t.z += v.z; t.w += v.w; }
            *reinterpret_cast<float4*>(red + o) = t;
        }
    }
    // scalars: [slot][kScal] doubles from up to ~750 CTAs.  Warp w adds the slots b = w, w + 8, ... (coalesced rows, four rows of
    // independent loads in flight), then the eight warp sums are added in warp order: a fixed order, and ~10x less latency than one
    // thread per scalar walking all slots.
    __shared__ double sc_s[8][kScal];
    if ((what & 2) && blockIdx.x == 0) {
        double acc[3] = {0.0, 0.0, 0.0};
        int b = w;
        for (; b + 24 < nslots; b += 32) {
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const int i = lane + 32 * c;
                if (i < kScal) {
                    const double v0 = Spart[(long long)b * kScal + i], v1 = Spart[(long long)(b + 8) * kScal + i];
                    const double v2 = Spart[(long long)(b + 16) * kScal + i], v3 = Spart[(long long)(b + 24) * kScal + i];
                    acc[c] = (((acc[c] + v0) + v1) + v2) + v3;
                }
            }
        }
        for (; b < nslots; b += 8)
#pragma unroll
            for (int c = 0; c < 3; ++c)
                if (lane + 32 * c < kScal) acc[c] += Spart[(long long)b * kScal + lane + 32 * c];
#pragma unroll
        for (int c = 0; c < 3; ++c)
            if (lane + 32 * c < kScal) sc_s[w][lane + 32 * c] = acc[c];
        __syncthreads();
    }
    if ((what & 2) && blockIdx.x == 0 && threadIdx.x < kScal) {
        const int i = threadIdx.x;
        double s = sc_s[0][i];
#pragma unroll
        for (int k = 1; k < 8; ++k) s += sc_s[k][i];
        // compact layout: [loss | gram r*r | domega 3r]
        if (i == 0) {
            red[ecount] = (float)s;
        } else if (i < 1 + kMaxR * kMaxR) {
            const int gi = (i - 1) / kMaxR, gj = (i - 1) % kMaxR;
            if (gi < r && gj < r && gi <= gj) {
                red[ecount + 1 + gi * r + gj] = (float)s;
                red[ecount + 1 + gj * r + gi] = (float)s;
            }
        } else {
            const int w2 = i - 1 - kMaxR * kMaxR;
            if (w2 < 3 * r) red[ecount + 1 + r * r + w2] = (float)s;
        }
    }
}

void reduce_partials_launch(const float* Epart, int nx, long long ecount, const double* Spart, int nslots, int r, float* red, cudaStream_t st,
                            int what) {
    const unsigned grid = (what & 1) ? (unsigned)((ecount + 127) / 128) : 1u;
    reduce_partials_kernel<<<grid, 256, 0, st>>>(Epart, nx, ecount, Spart, nslots, r, red, what);
}

// Chain rule for a D matrix left in ws.Dacc by the tensor-core kernel (same kernel the chunked FFMA path uses).
int chain_rule_launch(const desmo_shape* s, const MonoTable& mt, int T, int Kp, const float* P, const float* phi, const float* omega, float* dphi,
                      const Workspace& ws, int slot_base, int* nslots, cudaStream_t st) {
    (void)Kp;
    FusedArgs a{};
    a.P = P; a.phi = phi; a.omega = omega; a.dphi = dphi; a.Spart = ws.Spart; a.Dacc = ws.Dacc;
    a.n = s->n; a.ld = s->ld; a.m = s->m; a.mld = s->mld; a.r = s->r; a.T = T; a.K = T + 3 * s->r;
    a.scale = (float)(2.0 / ((double)s->n_global * (double)s->m));
    a.mt = mt;
    {
        static int sms = 0;
        if (!sms) {
            int dev = 0;
            DESMO_CUDA(cudaGetDevice(&dev));
            DESMO_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        }
        cudaError_t err = cudaSuccess;
        if (chain_rule_reg_dispatch(a, slot_base, sms, nslots, st, &err)) {  // compile-time library: registers only
            DESMO_CUDA(err);
            return DESMO_OK;
        }
    }
    const long long ntiles = (a.ld + kTile - 1) / kTile;
    const int gc = (int)(ntiles < 296 ? ntiles : 296);  // persistent: two CTAs per SM
    DESMO_CUDA(chain_rule_dispatch(a, slot_base, gc, 0, st));
    *nslots = gc;
    return DESMO_OK;
}

template <int KP, class UT>
static int launch_fused(const FusedArgs& a, int sms, size_t smem_cap, cudaStream_t st, int* gx_out, int* nslots_out) {
    using L = FusedSmem<KP>;
    // smallest number of time chunks whose E chunk fits next to the staging buffers
    int nchunk = 1, mc = a.mld;
    while (L::bytes(mc) > smem_cap) {
        ++nchunk;
        mc = (((a.mld + nchunk - 1) / nchunk) + kBT - 1) / kBT * kBT;
        if (mc <= kBT) {
            set_error("fused_fp32: shape does not fit shared memory");
            return DESMO_ERR_UNSUPPORTED;
        }
    }
    nchunk = (a.mld + mc - 1) / mc;
    const long long ntiles = (a.ld + kTile - 1) / kTile;
    // small meshes (the script-sized cylinder cases are 16 tiles): split the time axis further so that every SM gets a CTA
    if (ntiles * nchunk < sms) {
        const int want = (int)std::min<long long>(sms / ntiles, a.mld / (4 * kBT));
        if (want > nchunk) {
            mc = (((a.mld + want - 1) / want) + kBT - 1) / kBT * kBT;
            nchunk = (a.mld + mc - 1) / mc;
        }
    }
    FusedArgs b = a;
    b.nchunk = nchunk;
    b.mc = mc;
    const int per_chunk = sms / nchunk > 0 ? sms / nchunk : 1;
    const int gx = (int)(ntiles < per_chunk ? ntiles : per_chunk);
    DESMO_CUDA(cudaFuncSetAttribute(fused_fp32_kernel<KP, UT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L::bytes(mc)));
    if (nchunk > 1) DESMO_CUDA(cudaMemsetAsync(b.Dacc, 0, sizeof(float) * (size_t)KP * a.ld, st));
    fused_event_record(0, st);
    fused_fp32_kernel<KP, UT><<<dim3(gx, nchunk), kTile, L::bytes(mc), st>>>(b);
    fused_event_record(1, st);
    DESMO_CUDA(cudaGetLastError());
    int nslots = gx * nchunk;
    if (nchunk > 1) {
        const int gc = (int)(ntiles < 256 ? ntiles : 256);
        DESMO_CUDA(chain_rule_dispatch(b, nslots, gc, 0, st));
        nslots += gc;
    }
    *gx_out = gx;
    *nslots_out = nslots;
    return DESMO_OK;
}

template <int KP>
static int launch_fused_u(const FusedArgs& a, int u_dtype, int sms, size_t smem_cap, cudaStream_t st, int* gx_out, int* nslots_out) {
    return u_dtype == DESMO_DTYPE_BF16 ? launch_fused<KP, __nv_bfloat16>(a, sms, smem_cap, st, gx_out, nslots_out)
                                       : launch_fused<KP, float>(a, sms, smem_cap, st, gx_out, nslots_out);
}

int fused_fp32(const desmo_shape* s, const MonoTable& mt, int T, int Kp, const void* U, int u_dtype, const float* P, const float* phi,
               const float* omega, const float* W, float* dphi, float* red, const Workspace& ws, cudaStream_t st, bool supplied) {
    int dev = 0, sms = 0, smem_cap = 0;
    DESMO_CUDA(cudaGetDevice(&dev));
    DESMO_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    DESMO_CUDA(cudaDeviceGetAttribute(&smem_cap, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    FusedArgs a{};
    a.U = U; a.P = P; a.phi = phi; a.omega = omega; a.W = W; a.dphi = dphi;
    a.Epart = ws.Epart; a.Spart = ws.Spart; a.Dacc = ws.Dacc;
    a.n = s->n; a.ld = s->ld; a.m = s->m; a.mld = s->mld; a.r = s->r; a.T = T; a.K = T + 3 * s->r;
    a.scale = (float)(2.0 / ((double)s->n_global * (double)s->m));
    a.seed_scale = supplied ? (float)(0.5 * (double)s->n_global * (double)s->m) : 0.0f;
    a.mt = mt;
    int gx = 0, nslots = 0, rc = 0;
    switch (Kp) {
        case 16: rc = launch_fused_u<16>(a, u_dtype, sms, smem_cap, st, &gx, &nslots); break;
        case 32: rc = launch_fused_u<32>(a, u_dtype, sms, smem_cap, st, &gx, &nslots); break;
        case 48: rc = launch_fused_u<48>(a, u_dtype, sms, smem_cap, st, &gx, &nslots); break;
        case 64: rc = launch_fused_u<64>(a, u_dtype, sms, smem_cap, st, &gx, &nslots); break;
        case 80: rc = launch_fused_u<80>(a, u_dtype, sms, smem_cap, st, &gx, &nslots); break;  // r = 8, p = 2 (K = 69): BASELINE's "8 modes"
        default: set_error("fused_fp32: padded K=%d not instantiated", Kp); return DESMO_ERR_UNSUPPORTED;
    }
    if (rc) return rc;
    const long long ecount = (long long)Kp * s->mld;
    reduce_partials_launch(ws.Epart, gx, ecount, ws.Spart, nslots, s->r, red, st, 3);
    DESMO_CUDA(cudaGetLastError());
    return DESMO_OK;
}

}  // namespace desmo
